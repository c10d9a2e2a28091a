// Wasserstein barycenters of spectra (W2, 1-D): K rows of n bins per barycenter with weights λ -> the barycenter's
// mass at each point of an ascending output grid, and its gradient with respect to the rows.
//
// In 1-D the barycenter's quantile function is Σ_j λ_j Q_j.  Per barycenter, with c_j the CDF of row j:
//   cdf      the pairwise path's CDF pre-pass over the K rows (each normalised by its own mass; fp32 CDF, fp64 mass)
//   merge    ceil(log2 K) rounds (at least one) of two-run merge-path merges of the K CDF rows into their stable
//            order (row first, then bin, on equal values) as (value qs, label j * n + i) pairs
//   totals   per chunk of kChunk merged slots: the fp64 running sum of the increments of z (below)
//   scan     per barycenter, in chunk order: the running sum at every chunk start and at the start of the tie group
//            the chunk opens in; the poisoned-barycenter test (non-finite row, negative or non-finite weight)
//   walk     per chunk: Δ_k = qs_k - qs_{k-1} deposited at z_k onto the output grid by linear split (fp64 sums)
//   finish   per output point: the chunks' edge bins added in chunk order
// z of a tie group is Σ_j λ_j pos[min(lb_j, n - 1)], lb_j the entries of row j in front of the group.  Taking entry i of
// row j moves lb_j from i to i + 1, so z is a running sum S that starts at Σ_j λ_j pos[0] and adds the increments
// λ_j (pos[min(i + 1, n - 1)] - pos[i]) of the merged slots in front of the group; it is rounded to fp32 once per group.
// S has the same bits wherever it is formed: at a slot of chunk c it is fl(Z_c + P), P the chunk's own running sum from
// 0, Z_0 = Σ_j λ_j pos[0] and Z_{c+1} = fl(Z_c + P_end(c)), every operation rounded explicitly (no contraction).
// With λ >= 0 and ascending positions S never decreases, so neither do z and the output bin along the slots: a chunk's
// deposits fill a contiguous range of bins, the bins strictly inside it are stored by that chunk alone, and its two
// lowest and two highest bins are added by `finish`.
// Backward: dL/dqs_k = γ_k - γ_{k+1}, γ_k the upstream read back through slot k's split, written to the dL/dCDF entry
// slot k's label names (one writer per entry; a tie group shares z, so only its last slot is non-zero), then the
// pairwise path's per-row gradient arithmetic.  Every sum runs in a fixed order: two runs give the same bits, and a
// barycenter's result does not depend on the others in the call.
#include <cuda_runtime.h>

#include "../../include/sot_b200.h"
#include "sot_device.cuh"
#include "sot_internal.cuh"

namespace sot {
namespace barycenter {

constexpr int TPB = 256;
constexpr int kChunk = 512;                      // merged slots per walk thread
constexpr int kMergeSpan = 16;                   // output slots per merge thread
constexpr long long kMaxSlots = 1LL << 24;       // K x n per barycenter (labels and slot indices stay in int32)
constexpr long long kScratchBytes = 256LL << 20; // per wave of barycenters, unless one barycenter needs more

__host__ __device__ constexpr long long pad4(long long x) { return (x + 3) & ~3LL; }

struct Args {
    long long count;  // barycenters in this wave
    int k, n, m;      // rows per barycenter, bins per row, output points
    long long chunks; // walk chunks per barycenter
    const float* x;   // [count][k][n]
    const float* w;   // weights of barycenter b at w + b * w_stride
    long long w_stride;
    const float* pos;
    const float* pos_out;
    float* cdf;   // [count * k][pad4(n + 2)]
    double* mass; // [count * k]
    float* qv;    // [count][k * n] merged values
    int* ql;      // [count][k * n] merged labels
    double* tot;  // [count][chunks] P at the chunk's end
    double* open; // [count][chunks] P at the last tie-group start inside the chunk, -1 if there is none
    double* z0;   // [count][chunks] S at the chunk's first slot
    double* zg;   // [count][chunks] S at the start of the tie group of the chunk's first slot
    int* bad;     // [count] non-finite row or negative / non-finite weight: NaN results
    int* lo;      // [count][chunks] bin of the chunk's first slot
    int* hi;      // [count][chunks] bin of its last slot + 1
    double* part; // [count][chunks][4] deposits into bins lo, lo + 1 (before the end) and hi - 1, hi (at the end)
};

// ---- merge: one round of two-run merges of runs of `run` slots (round 0 reads the CDF rows, label = slot) ---------
template <bool FIRST>
__global__ void __launch_bounds__(TPB) sot_barycenter_merge_kernel(const Args a, long long run,
                                                                   const float* __restrict__ iv,
                                                                   const int* __restrict__ il, float* __restrict__ ov,
                                                                   int* __restrict__ ol) {
    const long long T = static_cast<long long>(a.k) * a.n;
    const long long per = (T + kMergeSpan - 1) / kMergeSpan;
    const long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (t >= a.count * per) return;
    const long long b = t / per;
    const long long stride = pad4(a.n + 2);
    const float* const crow = a.cdf + b * a.k * stride;
    const float* const vin = iv + b * T;
    const int* const lin = il + b * T;
    auto val = [&](long long s) {
        if constexpr (FIRST) {
            const long long j = s / a.n;
            return crow[j * stride + (s - j * a.n)];
        } else {
            return vin[s];
        }
    };
    auto lab = [&](long long s) {
        if constexpr (FIRST) return static_cast<int>(s);
        else return lin[s];
    };
    long long d = (t - b * per) * kMergeSpan;
    const long long d_end = min(d + kMergeSpan, T);
    while (d < d_end) {
        const long long p0 = d / (2 * run) * (2 * run);  // the pair of runs [p0, p0 + la) and [p0 + la, p0 + la + lb)
        const long long la = min(run, T - p0), lb = min(run, T - p0 - la);
        const long long end = min(d_end, p0 + la + lb), diag = d - p0;
        long long lo = max(0LL, diag - lb), hi = min(diag, la);  // largest i with A[i-1] <= B[diag-i] (A first on ties)
        while (lo < hi) {
            const long long mid = (lo + hi + 1) >> 1;
            if (val(p0 + mid - 1) <= val(p0 + la + diag - mid)) lo = mid; else hi = mid - 1;
        }
        long long i = lo, j = diag - lo;
        for (; d < end; ++d) {
            const bool take_b = j < lb && (i >= la || val(p0 + la + j) < val(p0 + i));
            const long long s = take_b ? p0 + la + j : p0 + i;
            ov[b * T + d] = val(s);
            ol[b * T + d] = lab(s);
            if (take_b) ++j; else ++i;
        }
    }
}

// λ_j (pos[min(i + 1, n - 1)] - pos[i]) for the entry `label` = j * n + i; rounded the same way everywhere
SOT_DEVINL double increment(const Args& a, const float* lam, int label) {
    const int j = label / a.n, i = label - j * a.n;
    const double d = __dsub_rn(static_cast<double>(a.pos[min(i + 1, a.n - 1)]), static_cast<double>(a.pos[i]));
    return __dmul_rn(static_cast<double>(lam[j]), d);
}

// ---- totals: P at each chunk's end and at its last tie-group start ----------------------------------------------
__global__ void __launch_bounds__(TPB) sot_barycenter_totals_kernel(const Args a) {
    const long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (t >= a.count * a.chunks) return;
    const long long b = t / a.chunks, c = t - b * a.chunks;
    const long long T = static_cast<long long>(a.k) * a.n;
    const long long s0 = c * kChunk, s1 = min(s0 + kChunk, T);
    const float* const qv = a.qv + b * T;
    const int* const ql = a.ql + b * T;
    const float* const lam = a.w + b * a.w_stride;
    double P = 0.0, open = -1.0;
    for (long long s = s0; s < s1; ++s) {
        if (s == 0 || qv[s] != qv[s - 1]) open = P;
        P = __dadd_rn(P, increment(a, lam, ql[s]));
    }
    a.tot[t] = P;
    a.open[t] = open;
}

// ---- scan: one thread per barycenter, chunks in order --------------------------------------------------------------
__global__ void __launch_bounds__(TPB) sot_barycenter_scan_kernel(const Args a) {
    const long long b = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (b >= a.count) return;
    const long long T = static_cast<long long>(a.k) * a.n;
    const float* const lam = a.w + b * a.w_stride;
    const float* const qv = a.qv + b * T;
    bool bad = false;
    double z = 0.0;
    for (int j = 0; j < a.k; ++j) {
        const float l = lam[j];
        bad |= !(l >= 0.0f && isfinite(l)) || !isfinite(a.mass[b * a.k + j]);
        z = __dadd_rn(z, __dmul_rn(static_cast<double>(l), static_cast<double>(a.pos[0])));
    }
    a.bad[b] = bad;
    double group = z;  // S at the most recent tie-group start
    for (long long c = 0; c < a.chunks; ++c) {
        const long long q = b * a.chunks + c;
        const long long s0 = c * kChunk;
        if (s0 == 0 || qv[s0] != qv[s0 - 1]) group = z;
        a.z0[q] = z;
        a.zg[q] = group;
        const double o = a.open[q];
        if (o >= 0.0) group = __dadd_rn(z, o);
        z = __dadd_rn(z, a.tot[q]);
    }
}

// Bin b (in [0, M - 2]; 0 when M == 1) and the share f of bin b in the split of a unit mass at z; bin b + 1 gets
// 1 - f.  z below the grid goes to bin 0, z at or above its last point to bin M - 1.  `b` comes in as a lower bound of
// the answer (z never decreases along a chunk) and is advanced.
SOT_DEVINL double split(const float* po, int M, float z, int& b) {
    if (M == 1 || !(z >= po[0])) {
        b = 0;
        return 1.0;
    }
    if (z >= po[M - 1]) {
        b = M - 2;
        return 0.0;
    }
    while (po[b + 1] <= z) ++b;
    return (static_cast<double>(po[b + 1]) - z) / (static_cast<double>(po[b + 1]) - po[b]);
}

// largest b with po[b] <= z, clamped to [0, M - 2] (a start for `split`)
SOT_DEVINL int first_bin(const float* po, int M, float z) {
    int lo = 0, hi = M - 1;  // po[lo] <= z or lo == 0
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (po[mid] <= z) lo = mid; else hi = mid;
    }
    return max(0, min(lo, M - 2));
}

// ---- walk: one thread per chunk.  Forward: deposits; GRAD: dL/dCDF of every entry --------------------------------------
template <bool GRAD>
__global__ void __launch_bounds__(TPB) sot_barycenter_walk_kernel(const Args a, float* __restrict__ out,
                                                                  const float* __restrict__ up,
                                                                  float* __restrict__ dcdf) {
    const long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (t >= a.count * a.chunks) return;
    const long long b = t / a.chunks, c = t - b * a.chunks;
    const long long T = static_cast<long long>(a.k) * a.n;
    const long long s0 = c * kChunk, s1 = min(s0 + kChunk, T);
    const int M = a.m;
    if (a.bad[b]) {  // forward: `finish` writes the NaN row
        if constexpr (GRAD)
            for (long long s = s0; s < s1; ++s) dcdf[b * T + s] = f_nan();
        return;
    }
    const float* const qv = a.qv + b * T;
    const int* const ql = a.ql + b * T;
    const float* const lam = a.w + b * a.w_stride;
    const float* const po = a.pos_out;
    const double Z = a.z0[t];
    double P = 0.0, S = a.zg[t];  // S: z of the tie group open at the current slot, in fp64
    float prev = s0 > 0 ? qv[s0 - 1] : 0.0f;
    float zf = 0.0f;  // z of the current tie group
    int bin = 0;
    if constexpr (!GRAD) {
        int lo = -1, cur = 0;
        double a0 = 0.0, a1 = 0.0, p0 = 0.0, p1 = 0.0;
        float* const row = out + b * M;
        auto emit = [&](int mb, double v) {  // bins arrive in increasing order, each once
            if (mb == lo) p0 = v;
            else if (mb == lo + 1) p1 = v;
            else row[mb] = static_cast<float>(v);
        };
        for (long long s = s0; s < s1; ++s) {
            const float q = qv[s];
            if (s > s0 && q != prev) S = __dadd_rn(Z, P);
            if (s == s0 || q != prev) zf = static_cast<float>(S);
            if (s == s0) bin = first_bin(po, M, zf);
            const double f = split(po, M, zf, bin);
            if (lo < 0) lo = cur = bin;
            if (bin != cur) {
                emit(cur, a0);
                if (bin == cur + 1) {
                    a0 = a1;
                } else {
                    emit(cur + 1, a1);
                    for (int mb = cur + 2; mb < bin; ++mb) emit(mb, 0.0);
                    a0 = 0.0;
                }
                a1 = 0.0;
                cur = bin;
            }
            const double dq = static_cast<double>(q) - static_cast<double>(prev);
            a0 += dq * f;
            a1 += dq * (1.0 - f);
            P = __dadd_rn(P, increment(a, lam, ql[s]));
            prev = q;
        }
        a.lo[t] = lo;
        a.hi[t] = cur + 1;
        double* const pp = a.part + 4 * t;
        pp[0] = p0;
        pp[1] = p1;
        pp[2] = a0;
        pp[3] = a1;
    } else {
        const float* const g = up + b * M;
        auto gamma = [&](double f, int bb) {
            return static_cast<double>(g[bb]) * f + (M > 1 ? static_cast<double>(g[bb + 1]) * (1.0 - f) : 0.0);
        };
        double g_prev = 0.0;
        const long long last = s1 < T ? s1 : T - 1;  // slot s1 (the next chunk's first) only closes my last slot
        for (long long s = s0; s <= last; ++s) {
            const float q = qv[s];
            if (s > s0 && q != prev) S = __dadd_rn(Z, P);
            if (s == s0 || q != prev) zf = static_cast<float>(S);
            if (s == s0) bin = first_bin(po, M, zf);
            const double gk = gamma(split(po, M, zf, bin), bin);
            if (s > s0) dcdf[b * T + ql[s - 1]] = static_cast<float>(g_prev - gk);
            g_prev = gk;
            if (s == s1) break;
            P = __dadd_rn(P, increment(a, lam, ql[s]));
            prev = q;
        }
        if (s1 == T) dcdf[b * T + ql[T - 1]] = static_cast<float>(g_prev);  // γ past the last slot is 0
    }
}

// ---- finish: one thread per output point -----------------------------------------------------------------------------
__global__ void __launch_bounds__(TPB) sot_barycenter_finish_kernel(const Args a, float* __restrict__ out) {
    const long long t = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x;
    if (t >= a.count * a.m) return;
    const long long b = t / a.m;
    const int mb = static_cast<int>(t - b * a.m);
    if (a.bad[b]) {
        out[t] = f_nan();
        return;
    }
    const int* const lo = a.lo + b * a.chunks;
    const int* const hi = a.hi + b * a.chunks;
    long long c0 = 0, c1 = a.chunks;  // first chunk with hi >= mb (hi never decreases)
    while (c0 < c1) {
        const long long mid = (c0 + c1) >> 1;
        if (hi[mid] < mb) c0 = mid + 1; else c1 = mid;
    }
    double s = 0.0;
    for (long long c = c0; c < a.chunks && lo[c] <= mb; ++c) {
        if (mb >= lo[c] + 2 && mb <= hi[c] - 2) return;  // inside that chunk's range: it stored the bin itself
        const double* const pp = a.part + 4 * (b * a.chunks + c);
        if (mb == lo[c]) s += pp[0];
        if (mb == lo[c] + 1) s += pp[1];
        if (mb == hi[c] - 1) s += pp[2];
        if (mb == hi[c]) s += pp[3];
    }
    out[t] = static_cast<float>(s);
}

// Stream-ordered scratch carved into 256-byte aligned pieces.
struct Carve {
    long long bytes = 0;
    long long take(long long b) {
        const long long at = bytes;
        bytes += (b + 255) & ~255LL;
        return at;
    }
};

struct Layout {
    long long cdf, mass, qv[2], ql[2], tot, open, z0, zg, bad, lo, hi, part, dcdf, bytes;
};

Layout layout(long long count, int k, int n, long long chunks, bool grad) {
    const long long rows = count * k, T = count * k * static_cast<long long>(n), C = count * chunks;
    Carve c;
    Layout l{};
    l.cdf = c.take(4 * rows * pad4(n + 2));
    l.mass = c.take(8 * rows);
    for (int q = 0; q < 2; ++q) {
        l.qv[q] = c.take(4 * T);
        l.ql[q] = c.take(4 * T);
    }
    l.tot = c.take(8 * C);
    l.open = c.take(8 * C);
    l.z0 = c.take(8 * C);
    l.zg = c.take(8 * C);
    l.bad = c.take(4 * count);
    l.lo = c.take(4 * C);
    l.hi = c.take(4 * C);
    l.part = c.take(32 * C);
    l.dcdf = grad ? c.take(4 * T) : 0;
    l.bytes = c.bytes;
    return l;
}

unsigned blocks(long long items) { return static_cast<unsigned>((items + TPB - 1) / TPB); }

// One wave: `a.count` barycenters starting at x / weights already offset.  `out` [count][m] (forward) or
// `up` [count][m] and `grad` [count][k][n] (backward).
int run_wave(Args a, char* base, const Layout& l, bool square, float* out, const float* up, float* grad,
             cudaStream_t s) {
    const long long T = static_cast<long long>(a.k) * a.n;
    a.cdf = reinterpret_cast<float*>(base + l.cdf);
    a.mass = reinterpret_cast<double*>(base + l.mass);
    a.tot = reinterpret_cast<double*>(base + l.tot);
    a.open = reinterpret_cast<double*>(base + l.open);
    a.z0 = reinterpret_cast<double*>(base + l.z0);
    a.zg = reinterpret_cast<double*>(base + l.zg);
    a.bad = reinterpret_cast<int*>(base + l.bad);
    a.lo = reinterpret_cast<int*>(base + l.lo);
    a.hi = reinterpret_cast<int*>(base + l.hi);
    a.part = reinterpret_cast<double*>(base + l.part);
    const long long rows = a.count * a.k;
    int rc = pairwise::launch_row_cdfs(a.x, rows, a.n, square, a.cdf, a.mass, s);
    // merge rounds, ping-ponging between the two value / label buffers
    int src = 1;
    long long run = a.n;
    bool first = true;
    while (rc == SOT_OK && (first || run < T)) {
        const int dst = 1 - src;
        float* const ov = reinterpret_cast<float*>(base + l.qv[dst]);
        int* const ol = reinterpret_cast<int*>(base + l.ql[dst]);
        const float* const iv = reinterpret_cast<const float*>(base + l.qv[src]);
        const int* const il = reinterpret_cast<const int*>(base + l.ql[src]);
        const unsigned g = blocks(a.count * ((T + kMergeSpan - 1) / kMergeSpan));
        if (first) sot_barycenter_merge_kernel<true><<<g, TPB, 0, s>>>(a, run, iv, il, ov, ol);
        else sot_barycenter_merge_kernel<false><<<g, TPB, 0, s>>>(a, run, iv, il, ov, ol);
        rc = launched(cudaGetLastError(), "sot_barycenter_merge_kernel");
        src = dst;
        run *= 2;
        first = false;
    }
    a.qv = reinterpret_cast<float*>(base + l.qv[src]);
    a.ql = reinterpret_cast<int*>(base + l.ql[src]);
    const unsigned gc = blocks(a.count * a.chunks);
    if (rc == SOT_OK) {
        sot_barycenter_totals_kernel<<<gc, TPB, 0, s>>>(a);
        rc = launched(cudaGetLastError(), "sot_barycenter_totals_kernel");
    }
    if (rc == SOT_OK) {
        sot_barycenter_scan_kernel<<<blocks(a.count), TPB, 0, s>>>(a);
        rc = launched(cudaGetLastError(), "sot_barycenter_scan_kernel");
    }
    if (grad == nullptr) {
        if (rc == SOT_OK) {
            sot_barycenter_walk_kernel<false><<<gc, TPB, 0, s>>>(a, out, nullptr, nullptr);
            rc = launched(cudaGetLastError(), "sot_barycenter_walk_kernel");
        }
        if (rc == SOT_OK) {
            sot_barycenter_finish_kernel<<<blocks(a.count * a.m), TPB, 0, s>>>(a, out);
            rc = launched(cudaGetLastError(), "sot_barycenter_finish_kernel");
        }
        return rc;
    }
    float* const dcdf = reinterpret_cast<float*>(base + l.dcdf);
    if (rc == SOT_OK) {
        sot_barycenter_walk_kernel<true><<<gc, TPB, 0, s>>>(a, nullptr, up, dcdf);
        rc = launched(cudaGetLastError(), "sot_barycenter_walk_kernel");
    }
    if (rc == SOT_OK) rc = pairwise::launch_row_grads(a.x, rows, a.n, square, a.mass, dcdf, grad, s);
    return rc;
}

}  // namespace barycenter
}  // namespace sot

namespace {

using sot::fail;
namespace B = sot::barycenter;

int validate_barycenter(const sot_barycenter_problem* p) {
    if (p == nullptr) return fail(SOT_EINVAL, "problem is NULL");
    if (p->flags & ~SOT_SQUARE) return fail(SOT_EINVAL, "barycenters take SOT_SQUARE only");
    if (p->count < 0) return fail(SOT_EINVAL, "bad count %lld", (long long)p->count);
    if (p->count == 0) return SOT_OK;
    if (p->k < 1 || p->n < 1 || p->n_out < 1)
        return fail(SOT_EINVAL, "bad sizes: k=%d n=%d n_out=%d", p->k, p->n, p->n_out);
    if (static_cast<long long>(p->k) * p->n > B::kMaxSlots)
        return fail(SOT_ETOOBIG, "K x n = %lld entries per barycenter: the limit is %lld (2^24)",
                    static_cast<long long>(p->k) * p->n, B::kMaxSlots);
    if (p->weights_stride != 0 && p->weights_stride != p->k)
        return fail(SOT_EINVAL, "weights_stride must be 0 (shared weights) or k, got %lld", (long long)p->weights_stride);
    if (p->x == nullptr || p->weights == nullptr || p->pos == nullptr || p->pos_out == nullptr)
        return fail(SOT_EINVAL, "x, weights, pos or pos_out is NULL");
    return SOT_OK;
}

// Runs the barycenters in waves whose scratch stays within kScratchBytes (one barycenter at least); the scratch of
// the largest wave is allocated once, stream-ordered.
int run(const sot_barycenter_problem* p, float* out, const float* up, float* grad, cudaStream_t s) {
    const bool square = p->flags & SOT_SQUARE;
    const long long T = static_cast<long long>(p->k) * p->n, chunks = (T + B::kChunk - 1) / B::kChunk;
    const long long one = B::layout(1, p->k, p->n, chunks, grad != nullptr).bytes;
    long long wave = B::kScratchBytes / one;
    wave = wave < 1 ? 1 : (wave > p->count ? p->count : wave);
    const B::Layout l = B::layout(wave, p->k, p->n, chunks, grad != nullptr);
    char* scratch = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&scratch), static_cast<size_t>(l.bytes), s);
    if (e != cudaSuccess) return fail(static_cast<int>(e), "barycenter scratch: %s", cudaGetErrorString(e));
    int rc = SOT_OK;
    for (long long b0 = 0; b0 < p->count && rc == SOT_OK; b0 += wave) {
        B::Args a{};
        a.count = p->count - b0 < wave ? p->count - b0 : wave;
        a.k = p->k;
        a.n = p->n;
        a.m = p->n_out;
        a.chunks = chunks;
        a.x = p->x + b0 * T;
        a.w = p->weights + b0 * p->weights_stride;
        a.w_stride = p->weights_stride;
        a.pos = p->pos;
        a.pos_out = p->pos_out;
        rc = B::run_wave(a, scratch, l, square, out == nullptr ? nullptr : out + b0 * p->n_out,
                         up == nullptr ? nullptr : up + b0 * p->n_out, grad == nullptr ? nullptr : grad + b0 * T, s);
    }
    e = cudaFreeAsync(scratch, s);
    if (rc == SOT_OK && e != cudaSuccess) return fail(static_cast<int>(e), "cudaFreeAsync: %s", cudaGetErrorString(e));
    return rc;
}

}  // namespace

extern "C" {

int sot_barycenter_device(const sot_barycenter_problem* prob, float* out, void* stream) {
    if (int rc = validate_barycenter(prob)) return rc;
    if (prob->count == 0) return SOT_OK;
    if (out == nullptr) return fail(SOT_EINVAL, "out is NULL");
    return run(prob, out, nullptr, nullptr, static_cast<cudaStream_t>(stream));
}

int sot_barycenter_backward_device(const sot_barycenter_problem* prob, const float* upstream, float* grad_x,
                                   void* stream) {
    if (int rc = validate_barycenter(prob)) return rc;
    if (prob->count == 0) return SOT_OK;
    if (upstream == nullptr || grad_x == nullptr) return fail(SOT_EINVAL, "upstream or grad_x is NULL");
    return run(prob, nullptr, upstream, grad_x, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
