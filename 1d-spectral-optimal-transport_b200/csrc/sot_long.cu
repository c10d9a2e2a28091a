// Split-frame path: rows longer than one CTA's shared memory holds (real rows of more than 8448 bins), loss and
// gradients only.  `launch()` in sot_capi.cu takes it when no `kConfigs` entry fits the request, or when the
// override `sot_set_tuning(-1, 0, 0)` routes every row length here (tests and benchmarks).
//
// One CTA per frame, persistent grid.  The CDFs and dL/dCDF live in library-owned global scratch, one slot per CTA
// (allocated stream-ordered per launch, at most kScratchBytes unless a single frame needs more): a resident slice
// of frames keeps its re-reads in L2.  Per frame:
//   pass 0  masses: the fp64 carry of the per-tile sums of the CDF stage below (bitwise the same additions)
//   pass 1  CDFs, tile by tile (TPB threads x E bins): the entry arithmetic of stage 2 of sot_kernels.cuh -- packed
//           fp32 local prefixes, fp64 offsets (scan within the tile + carry across tiles), fp32 head / tail split of
//           offset * 1/mass, every entry capped by the next thread's head.  A tile's last thread is capped by the
//           next tile's first head (the same fp64 value), so the row is non-decreasing across tile borders, and the
//           row end is set to fl32(mass * 1/mass).  Raw weights: fp64 per entry, like the reference's CPU cumsum.
//   walk    merge-path co-rank search on the scratch CDFs, then each thread walks one chunk of the n + m merged
//           slots: sum dq * |dx|^p (searchsorted-left, clamp to the last bin, strict `qs > 1` mask).  Gradient
//           mode stores dL/dCDF at the last slot of each tie group (stable order, u before v) and patches groups
//           opened by an earlier chunk with a look-back over per-chunk carries (stage 3 of sot_kernels.cuh).
//   grad    mass term sum_i gw_i w_i (per thread S_t * P_t + sum_i ls_i w_i, over all tiles), then the tiles in
//           reverse: suffix sums of dL/dCDF (fp32 local, fp64 across threads and tiles), chain rule, x 2x, x upstream.
// Every reduction runs in a fixed order: two runs give the same bits.
#include <cuda_runtime.h>

#include <atomic>

#include "sot_launch.cuh"

namespace sot {
namespace longrow {

constexpr int TPB = 256;         // threads per frame
constexpr int E = 16;            // consecutive bins per thread and tile (one local prefix run: <= 3 ulp, DESIGN §4)
constexpr int TILE = TPB * E;
constexpr int NW = TPB / 32;
constexpr long long kScratchBytes = 64LL << 20;

__host__ __device__ constexpr long long pad4(long long x) { return (x + 3) & ~3LL; }

// floats of one CTA's scratch slot: CDF of u (n + 2 entries, two +inf sentinels), of v, then dL/dCDF (u then v)
__host__ __device__ constexpr long long slot_floats(int n, int m, bool grad) {
    return pad4(n + 2) + pad4(m + 2) + (grad ? pad4(static_cast<long long>(n) + m) : 0);
}

template <bool GRAD, bool RAW>
__global__ void __launch_bounds__(TPB) sot_long_kernel(const FrameArgs args, float* __restrict__ scratch) {
    __shared__ double red[6 * NW];  // scan slots (2 * NW), then the loss / dot partials of the warps
    __shared__ float carry[TPB];    // m*d of the tie group open at the end of each chunk (-1: none of its own)
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int n = args.n, m = args.m, K = n + m;
    const int rows = n > m ? n : m;
    const int ntiles = (rows + TILE - 1) / TILE;
    const bool square = args.flags & FLAG_SQUARE;
    const bool cut_scale = args.flags & FLAG_CUT_SCALE;
    const float thr = (args.flags & FLAG_LIMIT) ? 1.0f : FLT_BIG;
    const float p = args.p;
    float* const cu = scratch + static_cast<long long>(blockIdx.x) * slot_floats(n, m, GRAD);
    float* const cv = cu + pad4(n + 2);
    float* const g = cv + pad4(m + 2);  // [n + m]: dL/dCDF of u's entries, then of v's
    const int L = (K + TPB - 1) / TPB;  // merged slots per chunk, one chunk per thread
    const int k0 = min(tid * L, K), cnt = min(L, K - k0);
    double cta_loss = 0.0;

    for (long long frame = blockIdx.x; frame < args.n_frames; frame += gridDim.x) {
        const float* const xu = args.u + frame * n;
        const float* const xv = args.v + frame * m;
        const float* const pu = args.pos_u + frame * args.pos_u_stride;
        const float* const pv = args.pos_v + frame * args.pos_v_stride;
        // my E (u, v) bin pairs of the tile at t0 (zeros past the row ends)
        auto load = [&](int t0, f32x2 (&x2)[E]) {
            const int e0 = t0 + tid * E;
#pragma unroll
            for (int c = 0; c < E; ++c)
                x2[c] = pack2(e0 + c < n ? __ldg(xu + e0 + c) : 0.0f, e0 + c < m ? __ldg(xv + e0 + c) : 0.0f);
        };
        auto local_sum = [&](const f32x2 (&x2)[E]) {
            f32x2 t2 = 0;
            if (square) {
#pragma unroll
                for (int c = 0; c < E; ++c) t2 = fma2(x2[c], x2[c], t2);
            } else {
#pragma unroll
                for (int c = 0; c < E; ++c) t2 = add2(t2, x2[c]);
            }
            return t2;
        };
        auto raw_sums = [&](const f32x2 (&x2)[E], double& a, double& b) {
            a = b = 0.0;
#pragma unroll
            for (int c = 0; c < E; ++c) {
                float a_, b_;
                unpack2(x2[c], a_, b_);
                a += static_cast<double>(square ? a_ * a_ : a_);
                b += static_cast<double>(square ? b_ * b_ : b_);
            }
        };
        // exclusive fp64 offsets of my local sums within the tile, the next thread's, and the tile totals
        auto tile_scan = [&](const f32x2 (&x2)[E], double& ou, double& ov, double& nu, double& nv, double& tu,
                             double& tv) {
            if constexpr (RAW) {
                raw_sums(x2, ou, ov);
                cta_scan2d<TPB>(ou, ov, tu, tv, red, tid);
            } else {
                float Tu, Tv;
                unpack2(local_sum(x2), Tu, Tv);
                cta_scan2<TPB, false, true>(Tu, Tv, ou, ov, nu, nv, tu, tv, red, tid);
            }
            __syncthreads();  // (the scan slots are reused by the next tile)
        };

        // ---- pass 0: masses ----------------------------------------------------------------------------------
        double mass_u = 0.0, mass_v = 0.0;
        for (int t0 = 0; t0 < rows; t0 += TILE) {
            f32x2 x2[E];
            load(t0, x2);
            double ou, ov, nu = 0.0, nv = 0.0, tu, tv;
            tile_scan(x2, ou, ov, nu, nv, tu, tv);
            mass_u += tu;
            mass_v += tv;
        }
        const float mu32 = static_cast<float>(mass_u), mv32 = static_cast<float>(mass_v);
        bool u_live = mu32 > SAFE_EPS, v_live = mv32 > SAFE_EPS;  // utils.py:137
        double inv_u = recip_f64(u_live ? mu32 : SAFE_EPS);
        double inv_v = cut_scale ? inv_u : recip_f64(v_live ? mv32 : SAFE_EPS);
        if constexpr (RAW) {  // weights used as given: no normalisation, no mass term
            inv_u = inv_v = 1.0;
            u_live = v_live = false;
        }
        // NaN / inf anywhere (or an overflowing cut-mode scale) poisons the frame (CTA uniform)
        const bool finite = (fabs(mass_u * inv_u) <= static_cast<double>(FLT_BIG)) &&
                            (fabs(mass_v * inv_v) <= static_cast<double>(FLT_BIG));

        // ---- pass 1: CDFs ------------------------------------------------------------------------------------
        float acc = 0.0f;
        if (finite) {
            double car_u = 0.0, car_v = 0.0;
            for (int t0 = 0; t0 < rows; t0 += TILE) {
                f32x2 x2[E];
                load(t0, x2);
                double ou, ov, nu = 0.0, nv = 0.0, tu, tv;
                tile_scan(x2, ou, ov, nu, nv, tu, tv);
                const int e0 = t0 + tid * E;
                if constexpr (RAW) {
                    double ru = car_u + ou, rv = car_v + ov;
#pragma unroll
                    for (int c = 0; c < E; ++c) {
                        float a_, b_;
                        unpack2(x2[c], a_, b_);
                        ru += static_cast<double>(square ? a_ * a_ : a_);
                        rv += static_cast<double>(square ? b_ * b_ : b_);
                        if (e0 + c < n) cu[e0 + c] = static_cast<float>(ru);
                        if (e0 + c < m) cv[e0 + c] = static_cast<float>(rv);
                    }
                } else {
                    // offsets across tiles: carry + in-tile offset; the last thread's `next` is carry + tile total =
                    // the next tile's carry, i.e. bitwise the head the next tile's first thread starts from
                    const double base_u = (car_u + ou) * inv_u, base_v = (car_v + ov) * inv_v;
                    const float bh_u = static_cast<float>(base_u), bh_v = static_cast<float>(base_v);
                    const float bl_u = static_cast<float>(base_u - static_cast<double>(bh_u));
                    const float bl_v = static_cast<float>(base_v - static_cast<double>(bh_v));
                    const float cap_u = static_cast<float>((car_u + nu) * inv_u);
                    const float cap_v = static_cast<float>((car_v + nv) * inv_v);
                    const f32x2 bh2 = pack2(bh_u, bh_v), bl2 = pack2(bl_u, bl_v);
                    const f32x2 inv2 = pack2(static_cast<float>(inv_u), static_cast<float>(inv_v));
                    f32x2 p2 = 0;
#pragma unroll
                    for (int c = 0; c < E; ++c) {
                        p2 = square ? fma2(x2[c], x2[c], p2) : add2(p2, x2[c]);
                        float ca, cb;
                        unpack2(add2(fma2(p2, inv2, bl2), bh2), ca, cb);
                        if (e0 + c < n) cu[e0 + c] = fminf(ca, cap_u);
                        if (e0 + c < m) cv[e0 + c] = fminf(cb, cap_v);
                    }
                }
                car_u += tu;
                car_v += tv;
            }
            if (tid == 0) {
                cu[n] = cu[n + 1] = f_inf();  // sentinels (the second one is what the walk prefetches past the first)
                cv[m] = cv[m + 1] = f_inf();
            }
            __syncthreads();
            if constexpr (!RAW) {  // the row end is exact: fl32(mass * 1/mass) (never below the entry before it)
                if (tid == 0) cu[n - 1] = fmaxf(static_cast<float>(mass_u * inv_u), n > 1 ? cu[n - 2] : 0.0f);
                if (tid == 1) cv[m - 1] = fmaxf(static_cast<float>(mass_v * inv_v), m > 1 ? cv[m - 2] : 0.0f);
                __syncthreads();
            }

            // ---- walk: merge-path co-rank, then my chunk of merged slots ---------------------------------------
            int i, j;
            {
                int lo = max(0, k0 - m), hi = min(k0, n);  // largest i with cu[i-1] <= cv[k0-i] (u first on ties)
                while (lo < hi) {
                    const int mid = (lo + hi + 1) >> 1;
                    if (cu[mid - 1] <= cv[k0 - mid]) lo = mid; else hi = mid - 1;
                }
                i = lo;
                j = k0 - lo;
            }
            float a = cu[i], b = cv[j], an = cu[i + 1], bn = cv[j + 1];  // heads and the entries after them
            float pa = pu[min(i, n - 1)], pb = pv[min(j, m - 1)];
            float pan = pu[min(i + 1, n - 1)], pbn = pv[min(j + 1, m - 1)];
            float qprev = 0.0f;  // the zero the reference pads in front of qs (losses.py:301)
            if (k0 > 0) qprev = fmaxf(i > 0 ? cu[i - 1] : -f_inf(), j > 0 ? cv[j - 1] : -f_inf());
            int consumed = 0;  // index into g of the entry the last advance took
            auto advance = [&]() {
                if (b < a) {  // v (u first on equal values: the stable order of cat(cu, cv))
                    consumed = n + j;
                    ++j;
                    b = bn;
                    pb = pbn;
                    bn = cv[j + 1];
                    pbn = pv[min(j + 1, m - 1)];
                } else {
                    consumed = i;
                    ++i;
                    a = an;
                    pa = pan;
                    an = cu[i + 1];
                    pan = pu[min(i + 1, n - 1)];
                }
            };
            // the same accumulation in both kernels: the forward-only loss equals the fused one bit for bit
            auto accumulate = [&](float q, float D) { acc = fmaf(q > thr ? 0.0f : q - qprev, D, acc); };
            if constexpr (!GRAD) {
                for (int s = 0; s < cnt; ++s) {
                    const float q = fminf(a, b);
                    accumulate(q, cost_of_gap<0>(pa - pb, p));
                    qprev = q;
                    advance();
                }
            } else {
                // dL/dCDF = (m*d)_group - (m*d)_next group at a group's LAST slot, stored one step late (when the
                // next slot is known); a group that started before my chunk has unknown m*d: it is patched below
                constexpr int NO_FIX = -1;
                int fix = NO_FIX;
                float md_prev = 0.0f, carry_out = -1.0f;
                bool inherited = false;
                if (cnt > 0) {
                    const float q = fminf(a, b);
                    const float D = cost_of_gap<0>(pa - pb, p);
                    inherited = (k0 > 0) && (q == qprev);
                    md_prev = inherited ? 0.0f : (q > thr ? 0.0f : D);
                    accumulate(q, D);
                    qprev = q;
                    advance();
                    // slots 1 .. cnt, where slot cnt is the first of the next chunk (or the virtual slot K: both
                    // heads +inf, a new group with m*d = 0) and only closes my last group
                    for (int s = 1; s <= cnt; ++s) {
                        const float q2 = fminf(a, b);
                        const float D2 = cost_of_gap<0>(pa - pb, p);
                        const bool same = (q2 == qprev);
                        const float md = same ? md_prev : (q2 > thr ? 0.0f : D2);
                        g[consumed] = md_prev - md;
                        fix = (inherited && !same) ? consumed : fix;
                        inherited = inherited && same;
                        md_prev = md;
                        if (s == cnt) break;
                        accumulate(q2, D2);
                        qprev = q2;
                        advance();
                    }
                    carry_out = inherited ? -1.0f : md_prev;
                }
                carry[tid] = carry_out;
                __syncthreads();
                if (fix != NO_FIX) {  // look-back: chunk 0 never carries the marker
                    int t = tid - 1;
                    float c = carry[t];
                    while (c < 0.0f) c = carry[--t];
                    g[fix] += c;
                }
                __syncthreads();
            }
        }

        // ---- loss of the frame: fp32 chunk sums, added in fp64 in a fixed order -------------------------------
        double part = static_cast<double>(acc);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(FULL_MASK, part, off);
        if (lane == 0) red[2 * NW + wid] = part;
        __syncthreads();
        if (tid == 0) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < NW; ++k) s += red[2 * NW + k];
            const float frame_loss = finite ? static_cast<float>(s) : f_nan();
            if (args.loss != nullptr) args.loss[frame] = frame_loss;
            cta_loss += static_cast<double>(frame_loss);
        }
        __syncthreads();

        if constexpr (GRAD) {
            float* const ou = args.grad_u != nullptr ? args.grad_u + frame * n : nullptr;
            float* const ov = args.grad_v != nullptr ? args.grad_v + frame * m : nullptr;
            const float up = (args.upstream != nullptr ? args.upstream[frame] : 1.0f) *
                             (args.upstream_scale != nullptr ? *args.upstream_scale : 1.0f) * args.upstream_value;
            if (!finite) {
                for (int k = tid; k < n && ou != nullptr; k += TPB) ou[k] = f_nan();
                for (int k = tid; k < m && ov != nullptr; k += TPB) ov[k] = f_nan();
                continue;
            }
            auto gpair = [&](int e) { return pack2(e < n ? g[e] : 0.0f, e < m ? g[n + e] : 0.0f); };
            // ---- mass term: sum_i gw_i w_i = sum_t (S_t P_t + sum_i ls_i w_i), P_t = the CDF stage's prefix ----
            double dot_u = 0.0, dot_v = 0.0;
            if (u_live || v_live) {
                double car_u = 0.0, car_v = 0.0;
                for (int t0 = 0; t0 < rows; t0 += TILE) {
                    f32x2 x2[E];
                    load(t0, x2);
                    double ou_, ov_, nu = 0.0, nv = 0.0, tu, tv;
                    tile_scan(x2, ou_, ov_, nu, nv, tu, tv);
                    const int e0 = t0 + tid * E;
                    f32x2 s2 = 0, d2 = 0;
#pragma unroll
                    for (int c = E - 1; c >= 0; --c) {
                        s2 = add2(s2, gpair(e0 + c));
                        d2 = fma2(square ? mul2(x2[c], x2[c]) : x2[c], s2, d2);
                    }
                    float su, sv, du, dv;
                    unpack2(s2, su, sv);
                    unpack2(d2, du, dv);
                    dot_u += static_cast<double>(su) * (car_u + ou_) + static_cast<double>(du);
                    dot_v += static_cast<double>(sv) * (car_v + ov_) + static_cast<double>(dv);
                    car_u += tu;
                    car_v += tv;
                }
#pragma unroll
                for (int off = 16; off > 0; off >>= 1) {
                    dot_u += __shfl_xor_sync(FULL_MASK, dot_u, off);
                    dot_v += __shfl_xor_sync(FULL_MASK, dot_v, off);
                }
                if (lane == 0) {
                    red[2 * NW + wid] = dot_u;
                    red[3 * NW + wid] = dot_v;
                }
                __syncthreads();
                dot_u = dot_v = 0.0;
#pragma unroll
                for (int k = 0; k < NW; ++k) {
                    dot_u += red[2 * NW + k];
                    dot_v += red[3 * NW + k];
                }
                __syncthreads();
                dot_u *= inv_u;
                dot_v *= inv_v;
            }
            // a clamped mass has no derivative (torch.where picks the constant branch)
            const double corr_u = u_live ? (cut_scale ? dot_u + dot_v : dot_u) : 0.0;
            const double corr_v = (!cut_scale && v_live) ? dot_v : 0.0;
            const float ku = static_cast<float>(inv_u) * up * (square ? 2.0f : 1.0f);
            const float kv = static_cast<float>(inv_v) * up * (square ? 2.0f : 1.0f);
            const f32x2 k2 = pack2(ku, kv);
            // ---- tiles in reverse: suffix sums of dL/dCDF, chain rule, x 2x, x upstream --------------------------
            double suf_u = 0.0, suf_v = 0.0;  // sum of dL/dCDF of the tiles after this one
            for (int t = ntiles - 1; t >= 0; --t) {
                const int e0 = t * TILE + tid * E;
                f32x2 s2 = 0;
#pragma unroll
                for (int c = E - 1; c >= 0; --c) s2 = add2(s2, gpair(e0 + c));
                float su, sv;
                unpack2(s2, su, sv);
                double off_u, off_v, nu = 0.0, nv = 0.0, tu, tv;
                cta_scan2<TPB, true, false>(su, sv, off_u, off_v, nu, nv, tu, tv, red, tid);
                __syncthreads();
                const f32x2 b2 = pack2(static_cast<float>(suf_u + off_u - corr_u), static_cast<float>(suf_v + off_v - corr_v));
                suf_u += tu;
                suf_v += tv;
                f32x2 r2 = 0;
#pragma unroll
                for (int c = E - 1; c >= 0; --c) {
                    const int e = e0 + c;
                    r2 = add2(r2, gpair(e));
                    f32x2 o2 = mul2(add2(b2, r2), k2);
                    if (square)
                        o2 = mul2(o2, pack2(e < n ? __ldg(xu + e) : 0.0f, e < m ? __ldg(xv + e) : 0.0f));
                    float ga, gb;
                    unpack2(o2, ga, gb);
                    if (ou != nullptr && e < n) ou[e] = ga;
                    if (ov != nullptr && e < m) ov[e] = gb;
                }
            }
            __syncthreads();  // every read of g is done before the next frame's walk writes it
        }
    }
    if (tid == 0 && args.loss_sum != nullptr) {
        atomicAdd(args.loss_sum, cta_loss);  // one atomic per CTA
        if (args.ticket != nullptr) finish_mean(args);
    }
}

template <bool GRAD, bool RAW>
cudaError_t launch_kind(const FrameArgs& a, cudaStream_t stream) {
    auto kernel = sot_long_kernel<GRAD, RAW>;
    constexpr int kMaxDev = 64;  // resident CTAs of the chip, per device (see launch_one)
    static std::atomic<int> resident_of_dev[kMaxDev];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    int resident = (dev >= 0 && dev < kMaxDev) ? resident_of_dev[dev].load(std::memory_order_acquire) : 0;
    if (resident == 0) {
        int per_sm = 0, sms = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, TPB, 0);
        if (e != cudaSuccess) return e;
        e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return e;
        resident = (per_sm < 1 ? 1 : per_sm) * sms;
        if (dev >= 0 && dev < kMaxDev) resident_of_dev[dev].store(resident, std::memory_order_release);
    }
    const long long slot_bytes = 4LL * slot_floats(a.n, a.m, GRAD);
    long long grid = kScratchBytes / slot_bytes;
    if (grid < 1) grid = 1;
    if (grid > resident) grid = resident;
    if (grid > a.n_frames) grid = a.n_frames;
    // stream-ordered scratch: no host synchronisation, several streams may run the path at once, and a CUDA graph
    // that captures the launch captures the allocation with it
    float* scratch = nullptr;
    e = cudaMallocAsync(reinterpret_cast<void**>(&scratch), static_cast<size_t>(grid * slot_bytes), stream);
    if (e != cudaSuccess) return e;
    kernel<<<static_cast<unsigned>(grid), TPB, 0, stream>>>(a, scratch);
    const cudaError_t le = cudaGetLastError();
    e = cudaFreeAsync(scratch, stream);
    return le != cudaSuccess ? le : e;
}

}  // namespace longrow

cudaError_t sot_launch_long(const LaunchRequest& r, cudaStream_t stream) {
    const bool raw = r.args.flags & FLAG_RAW;
    if (r.out == OUT_GRAD)
        return raw ? longrow::launch_kind<true, true>(r.args, stream) : longrow::launch_kind<true, false>(r.args, stream);
    return raw ? longrow::launch_kind<false, true>(r.args, stream) : longrow::launch_kind<false, false>(r.args, stream);
}

}  // namespace sot
