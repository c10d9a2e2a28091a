// C ABI of libsot_b200.so (declared in include/sot_b200.h): argument validation, kernel
// configuration choice, and the host-buffer pipeline.  No torch types, no CPU compute path.
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#include "../../include/sot_b200.h"
#include "sot_launch.cuh"

// Production configurations (one per row-length class).  The alternatives that were only ever reachable through
// `sot_set_tuning` are compiled in with -DSOT_TUNING_CONFIGS (`SOT_BUILD_TUNING=1 python -m sot_b200.build`).
SOT_DECLARE_SUBWARP_CONFIG(16, 17, 280, 1)
SOT_DECLARE_CONFIG(32, 9, 296, 1)
SOT_DECLARE_CONFIG(64, 9, 584, 2)
SOT_DECLARE_CONFIG(32, 33, 1064, 1)
SOT_DECLARE_CONFIG(64, 17, 1096, 1)
SOT_DECLARE_CONFIG(128, 9, 1160, 1)
SOT_DECLARE_CONFIG(128, 17, 2184, 2)
SOT_DECLARE_CONFIG(256, 17, 4360, 2)
SOT_DECLARE_CONFIG(256, 33, 8456, 1)
#ifdef SOT_TUNING_CONFIGS
SOT_DECLARE_CONFIG(32, 9, 296, 2)
SOT_DECLARE_CONFIG(64, 17, 1096, 2)
SOT_DECLARE_CONFIG(32, 33, 1064, 2)
#endif

namespace sot {
// rows longer than shared memory holds (sot_long.cu)
cudaError_t sot_launch_long(const LaunchRequest& r, cudaStream_t stream);

// ------------------------------------------------------------------------------------------
// grad rows scaled by a per-frame factor: out[r, :] = unit[r, :] * s[r]   (backward of the
// "fused" mode, where the forward launch already produced d loss_r / d input)
// ------------------------------------------------------------------------------------------
// One warp per row (grid-stride over rows): the factor is read once per row, no per-element division; `out`
// may alias `unit`.
__global__ void __launch_bounds__(256) sot_scale_rows_kernel(const float* unit, const float* __restrict__ s,
                                                             float* out, long long rows, int width) {
    const int lane = threadIdx.x & 31;
    const long long warps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
    for (long long r = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5; r < rows; r += warps) {
        const float f = s[r];
        const float* src = unit + r * width;
        float* dst = out + r * width;
        for (int c = lane; c < width; c += 32) dst[c] = src[c] * f;
    }
}

// rows *= *scale, in place, for up to two buffers -- the whole backward of a step whose forward launch already
// produced the gradients of the mean (`sot_mean_step_device`).  The usual upstream gradient of a loss is exactly
// 1 (trainer.py:220,233-238: weight 1, `.mean()` of a scalar): every thread reads the scalar and leaves.
__global__ void __launch_bounds__(256) sot_scale_inplace_kernel(float* a, long long na, float* b, long long nb,
                                                                const float* __restrict__ scale) {
    const float f = *scale;
    if (f == 1.0f) return;
    const long long tid = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (int which = 0; which < 2; ++which) {
        float* p = which == 0 ? a : b;
        const long long n = which == 0 ? na : nb;
        if (p == nullptr || n <= 0) continue;
        // scalar head up to the first 16-byte boundary, float4 body, scalar tail
        const long long head = min(n, static_cast<long long>((16 - (reinterpret_cast<uintptr_t>(p) & 15)) & 15) >> 2);
        const long long body = (n - head) >> 2;
        float4* p4 = reinterpret_cast<float4*>(p + head);
        for (long long i = tid; i < body; i += stride) {
            float4 x = p4[i];
            x.x *= f;
            x.y *= f;
            x.z *= f;
            x.w *= f;
            p4[i] = x;
        }
        const long long done = head + 4 * body;
        if (tid < head) p[tid] *= f;
        if (tid < n - done) p[done + tid] *= f;
    }
}


// quantile_function (losses.py:214-220) as a stand-alone op: for every query level the position
// stored at the first CDF entry >= level (searchsorted 'left', index clamped to the last bin).
__global__ void __launch_bounds__(256) sot_quantile_lookup_kernel(const float* __restrict__ qs,
                                                                  const float* __restrict__ cws,
                                                                  const float* __restrict__ xs,
                                                                  float* __restrict__ out, long long rows, int k,
                                                                  int n) {
    const long long total = rows * k;
    const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
    for (long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; idx < total;
         idx += stride) {
        const long long r = idx / k;
        const float q = qs[idx];
        const float* row = cws + r * n;
        int lo = 0, hi = n;
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            if (row[mid] < q)
                lo = mid + 1;
            else
                hi = mid;
        }
        out[idx] = xs[r * n + min(lo, n - 1)];
    }
}

}  // namespace sot

namespace {

using LaunchFn = cudaError_t (*)(const sot::LaunchRequest&, cudaStream_t);
struct Config {
    int tpf, e, rs, nch;
    LaunchFn fn;
    bool sub;  // sub-warp frames (several frames per warp): real spectra -> loss / gradients only
    int max_bins() const { return tpf * e < rs - 7 ? tpf * e : rs - 7; }
};
// Ordered by preference for a given row length: the first entry that holds the row is used
// (choices from measurements on B200, profiles/).  Shared memory per CTA = (4 or 6) * 4 * rs bytes.
const Config kConfigs[] = {
    {16, 17, 280, 1, sot_launch_sub_16_17_280_1, true},  // <= 272 bins (n_fft 512: 257): two frames per warp
    {32, 9, 296, 1, sot_launch_32_9_296_1},      // <= 288 bins   (one warp per frame: plans, CDF harness, raw, complex)
    {64, 9, 584, 2, sot_launch_64_9_584_2},      // <= 576 bins   (n_fft 1024: 513)
    {32, 33, 1064, 1, sot_launch_32_33_1064_1},  // <= 1056 bins  (n_fft 2048: 1025): ONE WARP per frame, 33 bins per thread --
                                                 // no CTA barriers, half the per-frame fixed cost; since the gradient stage
                                                 // rebuilds its suffix sums (162 registers, no spills) 14 % faster than 64 x 17
    {64, 17, 1096, 1, sot_launch_64_17_1096_1},  // <= 1088 bins  (two warps per frame: the round-1 / early round-2 choice)
#ifdef SOT_TUNING_CONFIGS
    {32, 9, 296, 2, sot_launch_32_9_296_2},      // two-chain variant: measured slower
    {64, 17, 1096, 2, sot_launch_64_17_1096_2},  // alternatives for 1025 bins (profiles/r01j_tuning_experiments.txt)
    {32, 33, 1064, 2, sot_launch_32_33_1064_2},  // two merge chains per thread: 165 vs 182 M frames/s
#endif
    {128, 9, 1160, 1, sot_launch_128_9_1160_1},    // <= 1152 bins
    {128, 17, 2184, 2, sot_launch_128_17_2184_2},  // <= 2176 bins  (n_fft 4096: 2049)
    {256, 17, 4360, 2, sot_launch_256_17_4360_2},  // <= 4352 bins  (n_fft 8192: 4097)
    {256, 33, 8456, 1, sot_launch_256_33_8456_1},  // <= 8448 bins  (n_fft 16384: 8193)
};
constexpr int kNumConfigs = sizeof(kConfigs) / sizeof(kConfigs[0]);

thread_local char g_error[512] = "";
std::atomic<long long> g_launches{0};
std::atomic<int> g_tune_tpf{0}, g_tune_e{0}, g_tune_nch{0};
std::atomic<bool> g_prefer_sub{true};   // sub-warp configurations by default (when the request allows)
std::atomic<bool> g_force_long{false};  // sot_set_tuning(-1, 0, 0): every request the split-frame path serves takes it
constexpr int kMaxRowBins = (1 << 24) - 1;  // longest row (split-frame path)
constexpr int kMaxComplexBins = 4352;       // longest complex row: the two double-width landing rows fit shared memory

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_error, sizeof(g_error), fmt, ap);
    va_end(ap);
    return code;
}
int cuda_fail(cudaError_t e, const char* what) {
    snprintf(g_error, sizeof(g_error), "%s: %s", what, cudaGetErrorString(e));
    return static_cast<int>(e);
}

// `sub_ok`: the request is one the sub-warp configurations serve (see Config::sub)
const Config* pick_config(int n, int m, bool sub_ok = false) {
    const int need = n > m ? n : m;
    const int tt = g_tune_tpf.load(), te = g_tune_e.load();
    if (tt != 0) {
        for (int i = 0; i < kNumConfigs; ++i) {
            const Config& c = kConfigs[i];
            if (c.tpf == tt && c.e == te && (g_tune_nch.load() == 0 || c.nch == g_tune_nch.load()) &&
                c.max_bins() >= need && (!c.sub || sub_ok))
                return &c;
        }
    }
    for (int i = 0; i < kNumConfigs; ++i)
        if (kConfigs[i].max_bins() >= need && (!kConfigs[i].sub || (sub_ok && g_prefer_sub.load()))) return &kConfigs[i];
    return nullptr;
}

int validate(const sot_problem* p) {
    if (p == nullptr) return fail(SOT_EINVAL, "problem is NULL");
    if (p->n_frames < 0 || p->n_u < 1 || p->n_v < 1)
        return fail(SOT_EINVAL, "bad sizes: n_frames=%lld n_u=%d n_v=%d", (long long)p->n_frames, p->n_u, p->n_v);
    if (p->n_u > kMaxRowBins || p->n_v > kMaxRowBins)
        return fail(SOT_ETOOBIG, "rows longer than %d bins", kMaxRowBins);
    if (p->n_frames > 0 && (p->u == nullptr || p->v == nullptr)) return fail(SOT_EINVAL, "u or v is NULL");
    if (p->pos_u == nullptr || p->pos_v == nullptr)
        return fail(SOT_EINVAL, "support positions are required (pos_u / pos_v is NULL)");
    if (p->pos_u_stride < 0 || p->pos_v_stride < 0) return fail(SOT_EINVAL, "negative position stride");
    if (!(p->p >= 1.0f))  // also rejects NaN; losses.py:271
        return fail(SOT_EDOMAIN, "The OT loss is only valid for p>=1, %g was given", (double)p->p);
    if (p->flags & ~(SOT_SQUARE | SOT_CUT_SCALE | SOT_LIMIT | SOT_RAW_WEIGHTS | SOT_UNIFORM_GRID | SOT_COMPLEX_INPUT))
        return fail(SOT_EINVAL, "unknown flag bits");
    if ((p->n_frames + 3) / 4 > 0x7fffffffLL) return fail(SOT_ETOOBIG, "too many frames for one launch");
    return SOT_OK;
}

sot::FrameArgs base_args(const sot_problem* p) {
    sot::FrameArgs a;
    memset(&a, 0, sizeof(a));
    a.u = p->u;
    a.v = p->v;
    a.pos_u = p->pos_u;
    a.pos_v = p->pos_v;
    a.pos_u_stride = p->pos_u_stride;
    a.pos_v_stride = p->pos_v_stride;
    a.n_frames = p->n_frames;
    a.n = p->n_u;
    a.m = p->n_v;
    a.p = p->p;
    a.flags = p->flags;
    a.one = a.one_b = 1.0f;
    a.neg_zero = a.neg_zero_b = -0.0f;
    a.upstream_value = 1.0f;
    return a;
}

int launch(const sot_problem* p, sot::LaunchRequest& r, void* stream) {
    if ((p->flags & SOT_COMPLEX_INPUT) && (r.mode != sot::MODE_SPECTRA || r.out == sot::OUT_PLAN))
        return fail(SOT_EINVAL, "SOT_COMPLEX_INPUT is only valid for the forward / forward+backward entry points");
    if ((p->flags & SOT_COMPLEX_INPUT) && (p->flags & SOT_RAW_WEIGHTS))
        return fail(SOT_EINVAL, "SOT_RAW_WEIGHTS rows are real weights, not complex spectra");
    if (p->n_frames == 0) return SOT_OK;
    const bool sub_ok = r.mode == sot::MODE_SPECTRA && r.out != sot::OUT_PLAN &&
                        !(p->flags & (SOT_RAW_WEIGHTS | SOT_COMPLEX_INPUT)) && r.args.coranks_in == nullptr &&
                        r.args.coranks_out == nullptr;
    // the split-frame path (global-memory scratch): real rows, loss and gradients
    const bool long_ok = r.mode == sot::MODE_SPECTRA && r.out != sot::OUT_PLAN && !(p->flags & SOT_COMPLEX_INPUT);
    const Config* c = (long_ok && g_force_long.load()) ? nullptr : pick_config(p->n_u, p->n_v, sub_ok);
    // complex input keeps two double-width landing rows on top of the real rows: up to 10 rows of 4*rs bytes (+ pad, head)
    if ((p->flags & SOT_COMPLEX_INPUT) && (c == nullptr || 41 * c->rs + 8192 > 227 * 1024))
        return fail(SOT_ETOOBIG, "complex rows of %d / %d bins do not fit in shared memory (limit %d bins)", p->n_u,
                    p->n_v, kMaxComplexBins);
    if (c == nullptr && !long_ok)
        return fail(SOT_ETOOBIG, "rows of %d / %d bins exceed the largest kernel configuration of this entry point "
                    "(%d bins: quantile taps and the CDF harness run in shared memory)", p->n_u, p->n_v,
                    kConfigs[kNumConfigs - 1].max_bins());
    if (c == nullptr) {
        // Rows longer than shared memory holds run on the split-frame path, which re-reads its rows and positions from
        // global memory: it takes them only where the runtime confirms the device can reach them (a host buffer handed
        // to a device entry point, or no usable device, is refused here rather than faulting in the kernel).
        const void* rows_and_positions[] = {p->u, p->v, p->pos_u, p->pos_v};
        for (const void* q : rows_and_positions) {
            cudaPointerAttributes attr;
            const cudaError_t pe = cudaPointerGetAttributes(&attr, q);
            if (pe != cudaSuccess || attr.devicePointer == nullptr) {
                if (pe != cudaSuccess) cudaGetLastError();  // (not sticky: leave no error behind for the caller)
                return fail(SOT_ETOOBIG,
                            "rows of %d / %d bins exceed shared memory (%d bins) and the split-frame path needs rows "
                            "and positions in device-accessible memory (%s)",
                            p->n_u, p->n_v, kConfigs[kNumConfigs - 1].max_bins(),
                            pe != cudaSuccess ? cudaGetErrorString(pe) : "a pointer the device cannot reach");
            }
        }
    }
    cudaError_t e = c != nullptr ? c->fn(r, static_cast<cudaStream_t>(stream))
                                 : sot::sot_launch_long(r, static_cast<cudaStream_t>(stream));
    if (e != cudaSuccess) return cuda_fail(e, "sot_frames_kernel launch");
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return SOT_OK;
}

}  // namespace

extern "C" {

int sot_abi_version(void) { return SOT_B200_ABI_VERSION; }
const char* sot_last_error(void) { return g_error; }
int64_t sot_launch_count(void) { return g_launches.load(); }
// shared with sot_mss.cu (not part of the public header)
int sot_mss_launch_count_add(void) { return static_cast<int>(g_launches.fetch_add(1, std::memory_order_relaxed)); }
int sot_mss_fail(int code, const char* msg) { return code < 0 ? fail(code, "%s", msg) : (snprintf(g_error, sizeof(g_error), "%s", msg), code); }

int sot_set_tuning(int32_t tpf, int32_t e, int32_t chains) {
    if (tpf == 0 && e == 0) {
        g_tune_tpf = 0;
        g_tune_e = 0;
        g_tune_nch = 0;
        g_force_long = false;
        return SOT_OK;
    }
    if (tpf == -1 && e == 0 && chains == 0) {
        g_force_long = true;
        return SOT_OK;
    }
    for (int i = 0; i < kNumConfigs; ++i)
        if (kConfigs[i].tpf == tpf && kConfigs[i].e == e && (chains == 0 || kConfigs[i].nch == chains)) {
            g_tune_tpf = tpf;
            g_tune_e = e;
            g_tune_nch = chains;
            return SOT_OK;
        }
    return fail(SOT_EINVAL, "no kernel configuration with %d threads per frame, %d bins per thread, %d chain(s)", tpf,
                e, chains);
}

int sot_max_bins(int32_t /*with_grad*/, int32_t /*shared_positions*/) { return kMaxRowBins; }

int sot_forward_device(const sot_problem* prob, float* loss, void* stream) {
    if (int rc = validate(prob)) return rc;
    if (loss == nullptr && prob->n_frames > 0) return fail(SOT_EINVAL, "loss is NULL");
    sot::LaunchRequest r{base_args(prob), sot::OUT_LOSS, sot::MODE_SPECTRA};
    r.args.loss = loss;
    return launch(prob, r, stream);
}

int sot_forward_backward_device(const sot_problem* prob, const float* upstream, float* loss, float* grad_u,
                                float* grad_v, void* stream) {
    if (int rc = validate(prob)) return rc;
    sot::LaunchRequest r{base_args(prob), sot::OUT_GRAD, sot::MODE_SPECTRA};
    r.args.upstream = upstream;
    r.args.loss = loss;
    r.args.grad_u = grad_u;
    r.args.grad_v = grad_v;
    return launch(prob, r, stream);
}

// One co-rank per merge chunk.  The chunk boundaries depend on the row lengths and on the NUMBER of chunks only
// (L = ceil((n_u + n_v) / chunks) | 1, chunk c starts at merged slot c * L), not on how many bins a thread holds: two
// configurations with the same threads x chains cut the merged grid identically, so co-ranks saved by one are valid
// for the other -- the count is the whole compatibility condition.
int sot_coranks_per_frame(int32_t n_u, int32_t n_v) {
    if (g_force_long.load()) return 0;  // (the split-frame path keeps no co-ranks)
    const Config* c = pick_config(n_u, n_v);
    return c == nullptr ? 0 : c->tpf * c->nch;
}

int sot_forward_sum_device(const sot_problem* prob, float* loss, double* loss_sum, uint16_t* coranks_out,
                           int32_t coranks_per_frame, void* stream) {
    if (int rc = validate(prob)) return rc;
    sot::LaunchRequest r{base_args(prob), sot::OUT_LOSS, sot::MODE_SPECTRA};
    r.args.loss = loss;
    r.args.loss_sum = loss_sum;
    if (coranks_out != nullptr) {
        if (coranks_per_frame != sot_coranks_per_frame(prob->n_u, prob->n_v))
            return fail(SOT_EINVAL, "coranks_per_frame = %d, this configuration needs %d", coranks_per_frame,
                        sot_coranks_per_frame(prob->n_u, prob->n_v));
        r.args.coranks_out = coranks_out;
    }
    return launch(prob, r, stream);
}

int sot_forward_backward_scaled_device(const sot_problem* prob, const float* upstream, const float* upstream_scale,
                                       const uint16_t* coranks_in, int32_t coranks_per_frame, float* loss,
                                       float* grad_u, float* grad_v, void* stream) {
    if (int rc = validate(prob)) return rc;
    sot::LaunchRequest r{base_args(prob), sot::OUT_GRAD, sot::MODE_SPECTRA};
    r.args.upstream = upstream;
    r.args.upstream_scale = upstream_scale;
    r.args.loss = loss;
    r.args.grad_u = grad_u;
    r.args.grad_v = grad_v;
    // co-ranks saved by a launch of another configuration are useless: search again instead
    if (coranks_in != nullptr && coranks_per_frame == sot_coranks_per_frame(prob->n_u, prob->n_v))
        r.args.coranks_in = coranks_in;
    return launch(prob, r, stream);
}

int sot_scale_rows_device(const float* unit, const float* scale, float* out, int64_t rows, int32_t width,
                          void* stream) {
    if (rows < 0 || width < 1) return fail(SOT_EINVAL, "bad sizes: rows=%lld width=%d", (long long)rows, width);
    if (rows == 0) return SOT_OK;
    if (unit == nullptr || scale == nullptr || out == nullptr) return fail(SOT_EINVAL, "NULL pointer");
    long long blocks = (rows + 7) / 8;  // one warp per row, eight rows per block
    if (blocks > 148LL * 8) blocks = 148LL * 8;
    sot::sot_scale_rows_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        unit, scale, out, rows, width);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "sot_scale_rows_kernel launch");
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return SOT_OK;
}

int sot_scale_inplace_device(float* rows_a, int64_t count_a, float* rows_b, int64_t count_b, const float* scale,
                             void* stream) {
    if (count_a < 0 || count_b < 0) return fail(SOT_EINVAL, "bad sizes: count_a=%lld count_b=%lld", (long long)count_a,
                                                (long long)count_b);
    if (scale == nullptr) return fail(SOT_EINVAL, "scale is NULL");
    if ((rows_a == nullptr || count_a == 0) && (rows_b == nullptr || count_b == 0)) return SOT_OK;
    const long long most = count_a > count_b ? count_a : count_b;
    long long blocks = (most / 4 + 255) / 256;
    if (blocks < 1) blocks = 1;
    if (blocks > 148LL * 8) blocks = 148LL * 8;
    sot::sot_scale_inplace_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        rows_a, rows_a != nullptr ? count_a : 0, rows_b, rows_b != nullptr ? count_b : 0, scale);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "sot_scale_inplace_kernel launch");
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return SOT_OK;
}

int sot_mean_step_device(const sot_problem* prob, const sot_mean_plan* plan, float* loss, float* grad_u, float* grad_v,
                         void* stream) {
    if (int rc = validate(prob)) return rc;
    if (plan == nullptr || plan->workspace == nullptr) return fail(SOT_EINVAL, "plan or plan->workspace is NULL");
    if (plan->post_world < 0 || plan->post_world > 16 || (plan->post_world > 0 && plan->post_mailboxes == nullptr) ||
        (plan->post_world > 0 && (plan->post_rank < 0 || plan->post_rank >= plan->post_world ||
                                  (plan->post_seq == 0 && plan->post_seq_device == nullptr))))
        return fail(SOT_EINVAL, "bad peer-mailbox description in the plan");
    if (prob->n_frames == 0) return fail(SOT_EINVAL, "sot_mean_step_device needs at least one frame");
    const bool grads = grad_u != nullptr || grad_v != nullptr;
    sot::LaunchRequest r{base_args(prob), grads ? sot::OUT_GRAD : sot::OUT_LOSS, sot::MODE_SPECTRA};
    r.args.loss = loss;
    r.args.grad_u = grad_u;
    r.args.grad_v = grad_v;
    r.args.upstream_value = plan->grad_scale;
    r.args.upstream_scale = plan->grad_scale_device;
    r.args.loss_sum = plan->workspace;
    r.args.ticket = reinterpret_cast<unsigned int*>(plan->workspace + 1);
    r.args.mean_out = plan->mean_out;
    r.args.mean_scale = plan->mean_scale;
    r.args.total_out = plan->total_out;
    r.args.post_count = plan->count_value;
    r.args.post_world = plan->post_world;
    r.args.post_rank = plan->post_rank;
    r.args.post_seq = plan->post_seq;
    r.args.post_seq_dev = reinterpret_cast<unsigned long long*>(plan->post_seq_device);
    for (int k = 0; k < plan->post_world; ++k) {
        if (plan->post_mailboxes[k] == nullptr) return fail(SOT_EINVAL, "NULL peer mailbox");
        r.args.post_mailbox[k] = static_cast<double*>(plan->post_mailboxes[k]);
    }
    return launch(prob, r, stream);
}

int sot_quantile_lookup_device(const float* qs, const float* cws, const float* xs, float* out, int64_t rows,
                               int32_t n_levels, int32_t n_bins, void* stream) {
    if (rows < 0 || n_levels < 1 || n_bins < 1) return fail(SOT_EINVAL, "bad sizes");
    if (rows == 0) return SOT_OK;
    if (qs == nullptr || cws == nullptr || xs == nullptr || out == nullptr) return fail(SOT_EINVAL, "NULL pointer");
    long long blocks = (rows * n_levels + 255) / 256;
    if (blocks > 148LL * 16) blocks = 148LL * 16;
    sot::sot_quantile_lookup_kernel<<<static_cast<unsigned>(blocks), 256, 0, static_cast<cudaStream_t>(stream)>>>(
        qs, cws, xs, out, rows, n_levels, n_bins);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return cuda_fail(e, "sot_quantile_lookup_kernel launch");
    g_launches.fetch_add(1, std::memory_order_relaxed);
    return SOT_OK;
}

int sot_quantiles_device(const sot_problem* prob, float* uq, float* vq, float* qs, float* cu, float* cv, int32_t* iu,
                         int32_t* iv, void* stream) {
    if (int rc = validate(prob)) return rc;
    sot::LaunchRequest r{base_args(prob), sot::OUT_PLAN, sot::MODE_SPECTRA};
    r.args.plan_uq = uq;
    r.args.plan_vq = vq;
    r.args.plan_qs = qs;
    r.args.plan_cu = cu;
    r.args.plan_cv = cv;
    r.args.plan_iu = iu;
    r.args.plan_iv = iv;
    return launch(prob, r, stream);
}

int sot_plan_from_cdf_device(const sot_problem* prob, float* uq, float* vq, float* qs, int32_t* iu, int32_t* iv,
                             void* stream) {
    if (int rc = validate(prob)) return rc;
    sot::LaunchRequest r{base_args(prob), sot::OUT_PLAN, sot::MODE_CDF};
    r.args.plan_uq = uq;
    r.args.plan_vq = vq;
    r.args.plan_qs = qs;
    r.args.plan_iu = iu;
    r.args.plan_iv = iv;
    return launch(prob, r, stream);
}

int sot_loss_from_cdf_device(const sot_problem* prob, float* loss, float* g_cu, float* g_cv, void* stream) {
    if (int rc = validate(prob)) return rc;
    const bool grads = (g_cu != nullptr) || (g_cv != nullptr);
    sot::LaunchRequest r{base_args(prob), grads ? sot::OUT_GRAD : sot::OUT_LOSS, sot::MODE_CDF};
    r.args.loss = loss;
    r.args.grad_u = g_cu;
    r.args.grad_v = g_cv;
    return launch(prob, r, stream);
}

// ------------------------------------------------------------------------------------------
// Host-buffer pipeline: frames are cut into chunks; chunk c+1's host->device copy, chunk c's
// kernel and chunk c-1's device->host copy overlap on three streams (PCIe is full duplex).
// Device buffers, streams and events live in a per-device workspace that is reused by later calls
// (allocation would otherwise cost more than the kernels).
// ------------------------------------------------------------------------------------------
}  // extern "C" (reopened below)

namespace {

constexpr int kSlots = 3;
constexpr int kMaxDevices = 16;

struct HostSlot {
    float *u = nullptr, *v = nullptr, *gu = nullptr, *gv = nullptr, *loss = nullptr, *up = nullptr, *pu = nullptr,
          *pv = nullptr;
    size_t cap_u = 0, cap_v = 0, cap_gu = 0, cap_gv = 0, cap_loss = 0, cap_up = 0, cap_pu = 0, cap_pv = 0;
    cudaEvent_t in_done = nullptr, k_done = nullptr, out_done = nullptr;
};
struct HostWorkspace {
    bool ready = false;
    size_t cap_dpu = 0, cap_dpv = 0;
    float *d_pu = nullptr, *d_pv = nullptr;
    // content of the shared support rows that are on the device already (re-sent only when they change)
    float *h_pu = nullptr, *h_pv = nullptr;
    size_t len_pu = 0, len_pv = 0;
    cudaStream_t s_in = nullptr, s_k = nullptr, s_out = nullptr;
    HostSlot slot[kSlots];
};
HostWorkspace g_ws[kMaxDevices];
std::mutex g_ws_mutex[kMaxDevices];  // one per device: ranks / threads driving different GPUs do not serialise

cudaError_t grow(float** p, size_t* cap, size_t bytes) {
    if (bytes <= *cap) return cudaSuccess;
    if (*p != nullptr) {
        cudaError_t e = cudaFree(*p);
        if (e != cudaSuccess) return e;
        *p = nullptr;
        *cap = 0;
    }
    cudaError_t e = cudaMalloc(p, bytes);
    if (e == cudaSuccess) *cap = bytes;
    return e;
}

// shared support row -> device, unless the same values are there already
cudaError_t sync_positions(float** dev, size_t* cap, float** shadow, size_t* len, const float* host, size_t n,
                           cudaStream_t stream) {
    if (*dev != nullptr && *shadow != nullptr && *len == n && memcmp(*shadow, host, 4 * n) == 0) return cudaSuccess;
    cudaError_t e = grow(dev, cap, 4 * n);
    if (e != cudaSuccess) return e;
    float* copy = static_cast<float*>(realloc(*shadow, 4 * n));
    if (copy == nullptr) return cudaErrorMemoryAllocation;
    memcpy(copy, host, 4 * n);
    *shadow = copy;
    *len = n;
    return cudaMemcpyAsync(*dev, copy, 4 * n, cudaMemcpyHostToDevice, stream);
}

// Device address of a host buffer the GPU can reach directly (pinned by cudaHostAlloc / cudaHostRegister under unified
// addressing), or nullptr: pageable memory, or a pointer the runtime does not know.
template <typename T>
T* mapped_device_pointer(T* host) {
    if (host == nullptr) return nullptr;
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, host) != cudaSuccess) {
        cudaGetLastError();  // (older runtimes report unknown pointers as an error: clear it)
        return nullptr;
    }
    if (attr.type != cudaMemoryTypeHost || attr.devicePointer == nullptr) return nullptr;
    return static_cast<T*>(const_cast<void*>(static_cast<const void*>(attr.devicePointer)));
}

void release(HostWorkspace& w) {
    for (int k = 0; k < kSlots; ++k) {
        HostSlot& s = w.slot[k];
        cudaFree(s.u);
        cudaFree(s.v);
        cudaFree(s.gu);
        cudaFree(s.gv);
        cudaFree(s.loss);
        cudaFree(s.up);
        cudaFree(s.pu);
        cudaFree(s.pv);
        if (s.in_done) cudaEventDestroy(s.in_done);
        if (s.k_done) cudaEventDestroy(s.k_done);
        if (s.out_done) cudaEventDestroy(s.out_done);
    }
    cudaFree(w.d_pu);
    cudaFree(w.d_pv);
    free(w.h_pu);
    free(w.h_pv);
    if (w.s_in) cudaStreamDestroy(w.s_in);
    if (w.s_k) cudaStreamDestroy(w.s_k);
    if (w.s_out) cudaStreamDestroy(w.s_out);
    w = HostWorkspace();
}

}  // namespace

extern "C" {

int sot_host_release(int32_t device) {
    if (device < 0 || device >= kMaxDevices) return fail(SOT_EINVAL, "bad device ordinal %d", device);
    std::lock_guard<std::mutex> lock(g_ws_mutex[device]);
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    release(g_ws[device]);
    return SOT_OK;
}

int sot_loss_grad_host(const sot_problem* hp, const float* upstream, float* loss, float* grad_u, float* grad_v,
                       int32_t device) {
    if (int rc = validate(hp)) return rc;
    if (device < 0 || device >= kMaxDevices) return fail(SOT_EINVAL, "bad device ordinal %d", device);
    // the staging buffers, copies and host offsets below are sized for real rows (4 bytes per bin)
    if (hp->flags & SOT_COMPLEX_INPUT)
        return fail(SOT_EINVAL, "SOT_COMPLEX_INPUT is not supported by the host-buffer entry point (device entries only)");
    std::lock_guard<std::mutex> lock(g_ws_mutex[device]);
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return cuda_fail(e, "cudaSetDevice");
    const long long N = hp->n_frames;
    if (N == 0) return SOT_OK;
    const int n = hp->n_u, m = hp->n_v;
    const bool want_grad = grad_u != nullptr || grad_v != nullptr;
    long long chunk_bytes = 32LL << 20;  // ~32 MiB of input per chunk; SOT_HOST_CHUNK_MIB overrides (tuning)
    if (const char* env = getenv("SOT_HOST_CHUNK_MIB")) {
        const long long mib = atoll(env);
        if (mib >= 1 && mib <= 4096) chunk_bytes = mib << 20;
    }
    long long chunk = chunk_bytes / (4LL * (n + m));
    chunk = (chunk / 4) * 4;
    if (chunk < 4) chunk = 4;
    if (chunk > N) chunk = ((N + 3) / 4) * 4;
    const bool su = hp->pos_u_stride == 0, sv = hp->pos_v_stride == 0;

    HostWorkspace& w = g_ws[device];
    int rc = SOT_OK;
    // Zero-copy (SOT_HOST_ZEROCOPY=1; shared supports; every buffer pinned and mapped): ONE launch over the whole batch
    // whose bulk loads and stores go over PCIe themselves -- no staging buffers, no fill and drain of a copy pipeline.
    // Anything else (pageable memory, per-frame supports) takes the chunked pipeline below.
    // (rows longer than shared memory holds: the split-frame path re-reads its rows, so they are staged on the device)
    if (const char* zc = getenv("SOT_HOST_ZEROCOPY");
        zc != nullptr && zc[0] == '1' && su && sv && !g_force_long.load() && pick_config(n, m) != nullptr) {
        const float* du = mapped_device_pointer(hp->u);
        const float* dv = mapped_device_pointer(hp->v);
        const float* dup = mapped_device_pointer(upstream);
        float* dl = mapped_device_pointer(loss);
        float* dgu = mapped_device_pointer(grad_u);
        float* dgv = mapped_device_pointer(grad_v);
        const bool all_mapped = du != nullptr && dv != nullptr && (upstream == nullptr || dup != nullptr) &&
                                (loss != nullptr && dl != nullptr) && (grad_u == nullptr || dgu != nullptr) &&
                                (grad_v == nullptr || dgv != nullptr);
        if (all_mapped) {
            if (w.s_k == nullptr) {
                e = cudaStreamCreateWithFlags(&w.s_k, cudaStreamNonBlocking);
                if (e != cudaSuccess) return cuda_fail(e, "cudaStreamCreateWithFlags");
            }
            e = sync_positions(&w.d_pu, &w.cap_dpu, &w.h_pu, &w.len_pu, hp->pos_u, n, w.s_k);
            if (e == cudaSuccess) e = sync_positions(&w.d_pv, &w.cap_dpv, &w.h_pv, &w.len_pv, hp->pos_v, m, w.s_k);
            if (e != cudaSuccess) return cuda_fail(e, "sync_positions");
            sot_problem dp = *hp;
            dp.u = du;
            dp.v = dv;
            dp.pos_u = w.d_pu;
            dp.pos_v = w.d_pv;
            rc = want_grad ? sot_forward_backward_device(&dp, dup, dl, dgu, dgv, w.s_k) : sot_forward_device(&dp, dl, w.s_k);
            e = cudaStreamSynchronize(w.s_k);
            if (rc == SOT_OK && e != cudaSuccess) rc = cuda_fail(e, "cudaStreamSynchronize");
            return rc;
        }
    }
    constexpr int kTraceChunks = 64;
    const bool trace = getenv("SOT_HOST_TRACE") != nullptr;
    cudaEvent_t tev[4 * kTraceChunks] = {};
    long long n_traced = 0;
    if (trace)
        for (int k = 0; k < 4 * kTraceChunks; ++k) cudaEventCreate(&tev[k]);
#define SOT_CK(call)                             \
    do {                                         \
        cudaError_t _e = (call);                 \
        if (_e != cudaSuccess && rc == SOT_OK) { \
            rc = cuda_fail(_e, #call);           \
            goto done;                           \
        }                                        \
    } while (0)
    {
        if (!w.ready) {
            if (w.s_in == nullptr) SOT_CK(cudaStreamCreateWithFlags(&w.s_in, cudaStreamNonBlocking));
            if (w.s_k == nullptr) SOT_CK(cudaStreamCreateWithFlags(&w.s_k, cudaStreamNonBlocking));  // (zero-copy calls make it too)
            if (w.s_out == nullptr) SOT_CK(cudaStreamCreateWithFlags(&w.s_out, cudaStreamNonBlocking));
            for (int k = 0; k < kSlots; ++k) {
                SOT_CK(cudaEventCreateWithFlags(&w.slot[k].in_done, cudaEventDisableTiming));
                SOT_CK(cudaEventCreateWithFlags(&w.slot[k].k_done, cudaEventDisableTiming));
                SOT_CK(cudaEventCreateWithFlags(&w.slot[k].out_done, cudaEventDisableTiming));
            }
            w.ready = true;
        }
        if (su) SOT_CK(sync_positions(&w.d_pu, &w.cap_dpu, &w.h_pu, &w.len_pu, hp->pos_u, n, w.s_in));
        if (sv) SOT_CK(sync_positions(&w.d_pv, &w.cap_dpv, &w.h_pv, &w.len_pv, hp->pos_v, m, w.s_in));
        for (int k = 0; k < kSlots; ++k) {
            HostSlot& s = w.slot[k];
            SOT_CK(grow(&s.u, &s.cap_u, 4ULL * chunk * n));
            SOT_CK(grow(&s.v, &s.cap_v, 4ULL * chunk * m));
            SOT_CK(grow(&s.loss, &s.cap_loss, 4ULL * chunk));
            if (upstream != nullptr) SOT_CK(grow(&s.up, &s.cap_up, 4ULL * chunk));
            if (grad_u != nullptr) SOT_CK(grow(&s.gu, &s.cap_gu, 4ULL * chunk * n));
            if (grad_v != nullptr) SOT_CK(grow(&s.gv, &s.cap_gv, 4ULL * chunk * m));
            if (!su) SOT_CK(grow(&s.pu, &s.cap_pu, 4ULL * chunk * n));
            if (!sv) SOT_CK(grow(&s.pv, &s.cap_pv, 4ULL * chunk * m));
        }
        long long c = 0;
        for (long long f0 = 0; f0 < N; f0 += chunk, ++c) {
            HostSlot& s = w.slot[c % kSlots];
            const long long nf = (N - f0 < chunk) ? (N - f0) : chunk;
            if (c >= kSlots) SOT_CK(cudaStreamWaitEvent(w.s_in, s.out_done, 0));  // slot drained
            if (trace && c < kTraceChunks) SOT_CK(cudaEventRecord(tev[4 * c + 0], w.s_in));
            SOT_CK(cudaMemcpyAsync(s.u, hp->u + f0 * n, 4ULL * nf * n, cudaMemcpyHostToDevice, w.s_in));
            SOT_CK(cudaMemcpyAsync(s.v, hp->v + f0 * m, 4ULL * nf * m, cudaMemcpyHostToDevice, w.s_in));
            if (upstream != nullptr)
                SOT_CK(cudaMemcpyAsync(s.up, upstream + f0, 4ULL * nf, cudaMemcpyHostToDevice, w.s_in));
            if (!su)
                SOT_CK(cudaMemcpy2DAsync(s.pu, 4ULL * n, hp->pos_u + f0 * hp->pos_u_stride, 4ULL * hp->pos_u_stride,
                                         4ULL * n, nf, cudaMemcpyHostToDevice, w.s_in));
            if (!sv)
                SOT_CK(cudaMemcpy2DAsync(s.pv, 4ULL * m, hp->pos_v + f0 * hp->pos_v_stride, 4ULL * hp->pos_v_stride,
                                         4ULL * m, nf, cudaMemcpyHostToDevice, w.s_in));
            SOT_CK(cudaEventRecord(s.in_done, w.s_in));
            if (trace && c < kTraceChunks) SOT_CK(cudaEventRecord(tev[4 * c + 1], w.s_in));
            SOT_CK(cudaStreamWaitEvent(w.s_k, s.in_done, 0));
            sot_problem dp = *hp;
            dp.n_frames = nf;
            dp.u = s.u;
            dp.v = s.v;
            dp.pos_u = su ? w.d_pu : s.pu;
            dp.pos_v = sv ? w.d_pv : s.pv;
            dp.pos_u_stride = su ? 0 : n;
            dp.pos_v_stride = sv ? 0 : m;
            const int krc = want_grad ? sot_forward_backward_device(&dp, upstream != nullptr ? s.up : nullptr, s.loss,
                                                                    grad_u != nullptr ? s.gu : nullptr,
                                                                    grad_v != nullptr ? s.gv : nullptr, w.s_k)
                                      : sot_forward_device(&dp, s.loss, w.s_k);
            if (krc != SOT_OK) {
                rc = krc;
                goto done;
            }
            SOT_CK(cudaEventRecord(s.k_done, w.s_k));
            SOT_CK(cudaStreamWaitEvent(w.s_out, s.k_done, 0));
            if (trace && c < kTraceChunks) SOT_CK(cudaEventRecord(tev[4 * c + 2], w.s_out));
            if (loss != nullptr) SOT_CK(cudaMemcpyAsync(loss + f0, s.loss, 4ULL * nf, cudaMemcpyDeviceToHost, w.s_out));
            if (grad_u != nullptr)
                SOT_CK(cudaMemcpyAsync(grad_u + f0 * n, s.gu, 4ULL * nf * n, cudaMemcpyDeviceToHost, w.s_out));
            if (grad_v != nullptr)
                SOT_CK(cudaMemcpyAsync(grad_v + f0 * m, s.gv, 4ULL * nf * m, cudaMemcpyDeviceToHost, w.s_out));
            SOT_CK(cudaEventRecord(s.out_done, w.s_out));
            if (trace && c < kTraceChunks) SOT_CK(cudaEventRecord(tev[4 * c + 3], w.s_out));
        }
        n_traced = c < kTraceChunks ? c : kTraceChunks;
    }
done:
    // drain everything that was queued (also on the error path) before the host buffers are reused
    if (w.s_out) cudaStreamSynchronize(w.s_out);
    if (w.s_k) cudaStreamSynchronize(w.s_k);
    if (w.s_in) cudaStreamSynchronize(w.s_in);
    if (trace) {  // SOT_HOST_TRACE=1: when each chunk's H2D / D2H copies started and ended (ms since the first copy)
        for (long long k = 0; k < n_traced && rc == SOT_OK; ++k) {
            float t[4] = {0, 0, 0, 0};
            for (int j = 0; j < 4; ++j) cudaEventElapsedTime(&t[j], tev[0], tev[4 * k + j]);
            fprintf(stderr, "sot_loss_grad_host chunk %lld: h2d %.3f..%.3f  d2h %.3f..%.3f ms\n", k, t[0], t[1], t[2], t[3]);
        }
        for (int k = 0; k < 4 * kTraceChunks; ++k)
            if (tev[k]) cudaEventDestroy(tev[k]);
    }
#undef SOT_CK
    return rc;
}

}  // extern "C"
