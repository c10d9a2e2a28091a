// Pairwise SOT distances: W_p^p of every row of u against every row of v of the same batch entry,
// [B, P, n] x [B, R, m] -> [B, P, R], and its gradients, without materialising the P x R pairs.
//
// A row's CDF depends on that row alone (cut mode: up to one scale, below), so the CDFs are built ONCE per row and
// the pairs only walk them:
//   cdf      one CTA per row index k: u row k and v row k as the two lanes of the split-frame path's CDF stage
//            (256 x 16 tiles, `normalise` / `cdf_scale` / `cdf_entries` of sot_device.cuh), each row normalised by its
//            own mass.  Writes the fp32 CDF (padded to 4 floats, two +inf sentinels) and the fp64 mass to scratch.
//   loss     one CTA per tile of T u-rows x T v-rows (bulk-copied into shared memory with the two position rows), one
//            warp per pair: merge-path co-rank search, then each lane walks its chunk of the n + m merged slots with
//            the split-frame walk (searchsorted-left, clamp to the last bin, strict `qs > 1` mask, u before v on ties).
//   grad     dL/dCDF of a pair is linear in its upstream value, so the chain rule runs once per ROW: a warp owns a row
//            and walks all its pairs, adding G_ij * dL/dCDF into the row's accumulator in shared memory (one sweep
//            with u-rows owned for grad_u, one with v-rows owned for grad_v).  The partner range is cut into slices
//            whose partial rows go to scratch; the row kernel adds the slices in order and runs the split-frame
//            gradient arithmetic (mass term, fp64 suffix sums, `mass_terms`, `grad_scale`, x 2x) once per row.
// Cut mode (v / mass of u): v's CDF is stored normalised by v's own mass; the pair walk scales it by the ratio of the
// pair's 1/M_u to that factor and ends it at the paired kernels' row end (`VScale` below).
// Every sum runs in a fixed order: two runs give the same bits.
#include <cuda_runtime.h>

#include <atomic>
#include <cmath>
#include <cub/device/device_radix_sort.cuh>

#include "../../include/sot_b200.h"
#include "sot_device.cuh"
#include "sot_internal.cuh"

namespace sot {
namespace pairwise {

constexpr int TPB = 256;  // CDF and row-gradient kernels: threads per row pair (the split-frame path's tiles)
constexpr int E = 16;
constexpr int TILE = TPB * E;
constexpr int NW = TPB / 32;
constexpr int kMaxBins = 8448;                 // the shared-memory kernels' longest row
constexpr int kSmemBudget = 110 * 1024;        // a tile this size leaves room for two CTAs per SM
constexpr int kMaxSmem = 227 * 1024;
constexpr long long kTargetCtas = 1024;        // gradient sweeps: CTAs per batch entry the partner range is sliced for

__host__ __device__ constexpr long long pad4(long long x) { return (x + 3) & ~3LL; }

struct Args {
    long long batch, rows_u, rows_v;
    int n, m;
    const float* u;
    const float* v;
    const float* pos_u;
    const float* pos_v;
    float p;
    int flags;
    float* cu;  // [batch * rows_u][pad4(n + 2)]: CDF rows of the pre-pass
    float* cv;  // [batch * rows_v][pad4(m + 2)]
    double* mass_u;
    double* mass_v;
    int tile;  // rows of each side per CTA tile
};

// ---- the split-frame path's row stage: u row k and v row k as the two lanes of packed pairs --------------------
struct RowPair {
    const float* xu;
    const float* xv;
    int n, m;  // 0 for a side without a row at this index
    bool square;
};

SOT_DEVINL void load_tile(const RowPair& r, int t0, int tid, f32x2 (&x2)[E]) {
    const int e0 = t0 + tid * E;
#pragma unroll
    for (int c = 0; c < E; ++c)
        x2[c] = pack2(e0 + c < r.n ? __ldg(r.xu + e0 + c) : 0.0f, e0 + c < r.m ? __ldg(r.xv + e0 + c) : 0.0f);
}

// exclusive fp64 offsets of my local sums within the tile, the next thread's, and the tile totals
SOT_DEVINL void tile_scan(const RowPair& r, const f32x2 (&x2)[E], double& ou, double& ov, double& nu, double& nv,
                          double& tu, double& tv, double* red, int tid) {
    f32x2 t2 = 0;
    if (r.square) {
#pragma unroll
        for (int c = 0; c < E; ++c) t2 = fma2(x2[c], x2[c], t2);
    } else {
#pragma unroll
        for (int c = 0; c < E; ++c) t2 = add2(t2, x2[c]);
    }
    float Tu, Tv;
    unpack2(t2, Tu, Tv);
    cta_scan2<TPB, false, true>(Tu, Tv, ou, ov, nu, nv, tu, tv, red, tid);
    __syncthreads();  // (the scan slots are reused by the next tile)
}

SOT_DEVINL void row_masses(const RowPair& r, double& mass_u, double& mass_v, double* red, int tid) {
    mass_u = mass_v = 0.0;
    for (int t0 = 0; t0 < (r.n > r.m ? r.n : r.m); t0 += TILE) {
        f32x2 x2[E];
        load_tile(r, t0, tid, x2);
        double ou, ov, nu = 0.0, nv = 0.0, tu, tv;
        tile_scan(r, x2, ou, ov, nu, nv, tu, tv, red, tid);
        mass_u += tu;
        mass_v += tv;
    }
}

__global__ void __launch_bounds__(TPB) sot_pairwise_cdf_kernel(const Args a) {
    __shared__ double red[2 * NW];
    const int tid = threadIdx.x;
    const long long k = blockIdx.x;
    const RowPair r{a.u + k * a.n, a.v + k * a.m, k < a.batch * a.rows_u ? a.n : 0, k < a.batch * a.rows_v ? a.m : 0,
                    (a.flags & FLAG_SQUARE) != 0};
    const int n = r.n, m = r.m;
    float* const cu = a.cu + k * pad4(a.n + 2);
    float* const cv = a.cv + k * pad4(a.m + 2);
    double mass_u, mass_v;
    row_masses(r, mass_u, mass_v, red, tid);
    const Norm nm = normalise<false>(mass_u, mass_v, false);
    double car_u = 0.0, car_v = 0.0;
    for (int t0 = 0; t0 < (n > m ? n : m); t0 += TILE) {
        f32x2 x2[E];
        load_tile(r, t0, tid, x2);
        double ou, ov, nu = 0.0, nv = 0.0, tu, tv;
        tile_scan(r, x2, ou, ov, nu, nv, tu, tv, red, tid);
        const int e0 = t0 + tid * E;
        const auto store_u = [&](int c, float x) { if (e0 + c < n) cu[e0 + c] = x; };
        const auto store_v = [&](int c, float x) { if (e0 + c < m) cv[e0 + c] = x; };
        const CdfScale ks = cdf_scale(car_u + ou, car_v + ov, car_u + nu, car_v + nv, nm);
        if (r.square) cdf_entries<true>(x2, ks, store_u, store_v); else cdf_entries<false>(x2, ks, store_u, store_v);
        car_u += tu;
        car_v += tv;
    }
    if (tid == 0) {
        if (n > 0) {
            cu[n] = cu[n + 1] = f_inf();
            a.mass_u[k] = mass_u;
        }
        if (m > 0) {
            cv[m] = cv[m + 1] = f_inf();
            a.mass_v[k] = mass_v;
        }
    }
    __syncthreads();
    // the row end is exact: fl32(mass * 1/mass) (never below the entry before it)
    if (tid == 0 && n > 0) cu[n - 1] = fmaxf(static_cast<float>(mass_u * nm.inv_u), n > 1 ? cu[n - 2] : 0.0f);
    if (tid == 1 && m > 0) cv[m - 1] = fmaxf(static_cast<float>(mass_v * nm.inv_v), m > 1 ? cv[m - 2] : 0.0f);
}

// ---- one pair, one warp --------------------------------------------------------------------------------------------
// Cut mode: the pair's view of v's CDF is the stored row (normalised by v's own mass) times
// r = fl32(inv_v / inv_own), the ratio of the pair's factor (1 / M_u) to the one the row was stored with; a positive
// scale keeps the row non-decreasing.  The row end is set to the paired kernels' own, fmaxf(fl32(M_v * inv_v), the
// entry before it), and the sentinels stay +inf.  (The stored row ends at fl32(M_v * inv_own), which is 1 only up to an
// ulp, so no single scale makes the end exact.)  For a v row identical to the u row the scale is exactly 1 and the two
// CDFs are the same bits: the diagonal of wasserstein_cdist(x, x, ...) is exactly 0, as on the paired path.
struct VScale {
    float r, end;
};
template <bool CUT>
SOT_DEVINL float vat(const float* cv, int j, int m, const VScale& s) {
    if constexpr (CUT) return j < m - 1 ? cv[j] * s.r : (j == m - 1 ? s.end : f_inf());
    else return cv[j];
}

// Norm of a pair and, in cut mode, the view of v's stored CDF `cv` (a scale of 1 otherwise).
template <bool CUT>
SOT_DEVINL Norm pair_norm(double mass_u, double mass_v, const float* cv, int m, VScale& s) {
    const Norm nm = normalise<false>(mass_u, mass_v, CUT);
    s = VScale{1.0f, 0.0f};
    if constexpr (CUT) {
        const Norm own = normalise<false>(mass_v, mass_v, false);
        s.r = static_cast<float>(nm.inv_v / own.inv_u);
        s.end = fmaxf(static_cast<float>(mass_v * nm.inv_v), m > 1 ? cv[m - 2] * s.r : 0.0f);
    }
    return nm;
}

struct PairRows {
    const float* cu;
    const float* cv;
    const float* pu;
    const float* pv;
    int n, m;
    VScale r;
    float p, thr;
};

// My chunk of the n + m merged slots (the split-frame walk with a warp for a CTA).  Returns my fp32 partial loss.
// GRAD: emit(entry, dL/dCDF) once for every entry of the pair (entry < n: u's, else n + index into v), then once more
// for an entry whose tie group opened in an earlier chunk (`carry`: 32 floats of the warp).
template <bool GRAD, bool CUT, typename Emit>
SOT_DEVINL float walk_pair(const PairRows& w, int lane, float* carry, const Emit& emit) {
    const float* const cu = w.cu;
    const float* const cv = w.cv;
    const float* const pu = w.pu;
    const float* const pv = w.pv;
    const int n = w.n, m = w.m, K = n + m;
    const VScale r = w.r;
    const float p = w.p, thr = w.thr;
    const int L = (K + 31) / 32;
    const int k0 = min(lane * L, K), cnt = min(L, K - k0);
    int i, j;
    {
        int lo = max(0, k0 - m), hi = min(k0, n);  // largest i with cu[i-1] <= cv[k0-i] (u first on ties)
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (cu[mid - 1] <= vat<CUT>(cv, k0 - mid, m, r)) lo = mid; else hi = mid - 1;
        }
        i = lo;
        j = k0 - lo;
    }
    float a = cu[i], b = vat<CUT>(cv, j, m, r), an = cu[i + 1], bn = vat<CUT>(cv, j + 1, m, r);
    float pa = pu[min(i, n - 1)], pb = pv[min(j, m - 1)];
    float pan = pu[min(i + 1, n - 1)], pbn = pv[min(j + 1, m - 1)];
    float qprev = 0.0f;  // the zero the reference pads in front of qs (losses.py:301)
    if (k0 > 0) qprev = fmaxf(i > 0 ? cu[i - 1] : -f_inf(), j > 0 ? vat<CUT>(cv, j - 1, m, r) : -f_inf());
    int consumed = 0;
    auto advance = [&]() {
        if (b < a) {  // v (u first on equal values: the stable order of cat(cu, cv))
            consumed = n + j;
            ++j;
            b = bn;
            pb = pbn;
            bn = vat<CUT>(cv, j + 1, m, r);
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
    float acc = 0.0f;
    auto accumulate = [&](float q, float D) { acc = fmaf(q > thr ? 0.0f : q - qprev, D, acc); };
    if constexpr (!GRAD) {
        for (int s = 0; s < cnt; ++s) {
            const float q = fminf(a, b);
            accumulate(q, cost_of_gap<0>(pa - pb, p));
            qprev = q;
            advance();
        }
    } else {
        constexpr int NO_FIX = -1;
        int fix = NO_FIX;
        float md_prev = 0.0f, carry_out = -1.0f;
        bool inherited = false;
        if (cnt > 0) {
            const float q = fminf(a, b);
            const float D = cost_of_gap<0>(pa - pb, p);
            inherited = (k0 > 0) && (q == qprev);
            md_prev = inherited ? 0.0f : (q > thr ? 0.0f : D);
            qprev = q;
            advance();
            // slots 1 .. cnt; slot cnt is the first of the next chunk (or the virtual slot K) and only closes my last group
            for (int s = 1; s <= cnt; ++s) {
                const float q2 = fminf(a, b);
                const float D2 = cost_of_gap<0>(pa - pb, p);
                emit(consumed, tie_step(q2, qprev, q2 > thr ? 0.0f : D2, consumed, md_prev, inherited, fix));
                if (s == cnt) break;
                qprev = q2;
                advance();
            }
            carry_out = inherited ? -1.0f : md_prev;
        }
        carry[lane] = carry_out;
        __syncwarp();
        if (fix != NO_FIX) emit(fix, look_back(lane - 1, 1, [&](int t) { return carry[t]; }));
        __syncwarp();
    }
    return acc;
}

// fp32 partial losses of the lanes, added in fp64 in a fixed order
SOT_DEVINL double warp_sum(double part) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(FULL_MASK, part, off);
    return part;
}

SOT_DEVINL float thr_of(int flags) { return (flags & FLAG_LIMIT) ? 1.0f : FLT_BIG; }

// bulk copies of `count` consecutive CDF rows of `stride` floats (16-byte multiples at 16-byte aligned addresses)
SOT_DEVINL void copy_rows(float* dst, const float* src, int count, long long stride, uint64_t* bar) {
    for (int q = 0; q < count; ++q) bulk_g2s(dst + q * stride, src + q * stride, static_cast<uint32_t>(4 * stride), bar);
}

// ---- loss: one CTA per (batch entry, tile of u rows, tile of v rows), one warp per pair ----------------------------
template <bool CUT>
__global__ void __launch_bounds__(256) sot_pairwise_loss_kernel(const Args a, float* __restrict__ dist) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int T = a.tile, n = a.n, m = a.m;
    const long long su = pad4(n + 2), sv = pad4(m + 2);
    float* const spu = reinterpret_cast<float*>(smem);
    float* const spv = spu + pad4(n);
    float* const scu = spv + pad4(m);
    float* const scv = scu + T * su;
    float* const carry = scv + T * sv;  // 32 floats per warp
    uint64_t* const bar = reinterpret_cast<uint64_t*>(carry + 32 * (blockDim.x / 32));
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, warps = blockDim.x >> 5;
    const long long tiles_u = (a.rows_u + T - 1) / T, tiles_v = (a.rows_v + T - 1) / T;
    long long blk = blockIdx.x;
    const long long tv = blk % tiles_v;
    blk /= tiles_v;
    const long long tu = blk % tiles_u, b = blk / tiles_u;
    const int cnt_u = static_cast<int>(min(static_cast<long long>(T), a.rows_u - tu * T));
    const int cnt_v = static_cast<int>(min(static_cast<long long>(T), a.rows_v - tv * T));
    const long long ru0 = b * a.rows_u + tu * T, rv0 = b * a.rows_v + tv * T;  // first rows of the tile
    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
        mbar_expect_tx(bar, static_cast<uint32_t>(4 * (cnt_u * su + cnt_v * sv)));
        copy_rows(scu, a.cu + ru0 * su, cnt_u, su, bar);
        copy_rows(scv, a.cv + rv0 * sv, cnt_v, sv, bar);
    }
    for (int k = tid; k < n; k += blockDim.x) spu[k] = a.pos_u[k];
    for (int k = tid; k < m; k += blockDim.x) spv[k] = a.pos_v[k];
    __syncthreads();
    mbar_wait(bar, 0);
    const float thr = thr_of(a.flags);
    for (int q = wid; q < cnt_u * cnt_v; q += warps) {
        const int il = q / cnt_v, jl = q - il * cnt_v;
        VScale r;
        const double mu = a.mass_u[ru0 + il], mv = a.mass_v[rv0 + jl];
        const Norm nm = pair_norm<CUT>(mu, mv, scv + jl * sv, m, r);
        const bool finite = finite_frame(mu, mv, nm);  // (warp uniform)
        float acc = 0.0f;
        if (finite)
            acc = walk_pair<false, CUT>(PairRows{scu + il * su, scv + jl * sv, spu, spv, n, m, r, a.p, thr}, lane,
                                        carry + 32 * wid, [](int, float) {});
        const double s = warp_sum(static_cast<double>(acc));
        if (lane == 0) dist[(ru0 + il) * a.rows_v + tv * T + jl] = finite ? static_cast<float>(s) : f_nan();
    }
}

// ---- gradient sweep: a warp owns a row (v rows when OWN_V, else u rows) and walks its pairs with one slice of the
// partner rows; part[slice][row][:] = sum_pairs G * dL/dCDF of the owned row (NaN when a pair is not finite) and, for
// u rows in cut mode, part_s[slice][row] = sum_pairs G * sum_l dL/dcv_l * cv_l (v's mass flows into u's in cut mode).
template <bool OWN_V, bool CUT>
__global__ void __launch_bounds__(256) sot_pairwise_grad_kernel(const Args a, const float* __restrict__ up,
                                                                float* __restrict__ part, double* __restrict__ part_s,
                                                                int slices) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int T = a.tile, n = a.n, m = a.m;
    const int n_own = OWN_V ? m : n;
    const long long s_own = pad4(n_own + 2), s_str = pad4((OWN_V ? n : m) + 2);
    const long long rows_own = OWN_V ? a.rows_v : a.rows_u, rows_str = OWN_V ? a.rows_u : a.rows_v;
    float* const spu = reinterpret_cast<float*>(smem);
    float* const spv = spu + pad4(n);
    float* const sown = spv + pad4(m);
    float* const sstr = sown + T * s_own;
    float* const sacc = sstr + T * s_str;
    float* const carry = sacc + T * pad4(n_own);
    uint64_t* const bar = reinterpret_cast<uint64_t*>(carry + 32 * T);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const long long tiles_own = (rows_own + T - 1) / T, tiles_str = (rows_str + T - 1) / T;
    long long blk = blockIdx.x;
    const int slice = static_cast<int>(blk % slices);
    blk /= slices;
    const long long to = blk % tiles_own, b = blk / tiles_own;
    const int cnt_own = static_cast<int>(min(static_cast<long long>(T), rows_own - to * T));
    const long long ro0 = b * rows_own + to * T;
    const float* const cdf_own = OWN_V ? a.cv : a.cu;
    const float* const cdf_str = OWN_V ? a.cu : a.cv;
    const long long st_lo = tiles_str * slice / slices, st_hi = tiles_str * (slice + 1) / slices;

    if (tid == 0) {
        mbar_init(bar, 1);
        fence_mbar_init();
        mbar_expect_tx(bar, static_cast<uint32_t>(4 * cnt_own * s_own));
        copy_rows(sown, cdf_own + ro0 * s_own, cnt_own, s_own, bar);
    }
    for (int k = tid; k < n; k += blockDim.x) spu[k] = a.pos_u[k];
    for (int k = tid; k < m; k += blockDim.x) spv[k] = a.pos_v[k];
    for (int k = tid; k < T * pad4(n_own); k += blockDim.x) sacc[k] = 0.0f;
    uint32_t phase = 0;
    __syncthreads();
    mbar_wait(bar, phase);
    phase ^= 1;

    float* const acc = sacc + wid * pad4(n_own);
    const float* const own_row = sown + wid * s_own;
    const long long row = ro0 + wid;  // global index of my owned row
    const float thr = thr_of(a.flags);
    double s_lane = 0.0;
    for (long long st = st_lo; st < st_hi; ++st) {
        const int cnt_str = static_cast<int>(min(static_cast<long long>(T), rows_str - st * T));
        const long long rs0 = b * rows_str + st * T;
        __syncthreads();  // every warp is done with the previous partner tile
        if (tid == 0) {
            fence_async_smem();
            mbar_expect_tx(bar, static_cast<uint32_t>(4 * cnt_str * s_str));
            copy_rows(sstr, cdf_str + rs0 * s_str, cnt_str, s_str, bar);
        }
        mbar_wait(bar, phase);
        phase ^= 1;
        if (wid >= cnt_own) continue;
        for (int jl = 0; jl < cnt_str; ++jl) {
            const long long gu = OWN_V ? rs0 + jl : row, gv = OWN_V ? row : rs0 + jl;  // global u and v row
            const float* const str_row = sstr + jl * s_str;
            VScale r;
            const double mu = a.mass_u[gu], mv = a.mass_v[gv];
            const Norm nm = pair_norm<CUT>(mu, mv, OWN_V ? own_row : str_row, m, r);
            // G[b, i, j]: u row gu = b * rows_u + i, v row gv = b * rows_v + j
            const float g = up[gu * a.rows_v + (gv - b * a.rows_v)];
            if (!finite_frame(mu, mv, nm)) {
                for (int e = lane; e < n_own; e += 32) acc[e] = f_nan();
                __syncwarp();
                continue;
            }
            const PairRows pr{OWN_V ? str_row : own_row, OWN_V ? own_row : str_row, spu, spv, n, m, r, a.p, thr};
            if constexpr (OWN_V) {
                // cut mode: dL/dy of the pair is 1/M_u * (suffix of dL/dcv), and 1/M_u depends on the partner
                const float w = CUT ? g * static_cast<float>(nm.inv_u) : g;
                walk_pair<true, CUT>(pr, lane, carry + 32 * wid, [&](int e, float d) {
                    if (e >= n) acc[e - n] = fmaf(w, d, acc[e - n]);
                });
            } else {
                walk_pair<true, CUT>(pr, lane, carry + 32 * wid, [&](int e, float d) {
                    if (e < n) {
                        acc[e] = fmaf(g, d, acc[e]);
                    } else if (CUT) {
                        s_lane += static_cast<double>(g * d) * static_cast<double>(vat<CUT>(pr.cv, e - n, m, r));
                    }
                });
            }
            __syncwarp();
        }
    }
    __syncthreads();
    if (wid < cnt_own) {
        float* const out = part + (slice * (a.batch * rows_own) + row) * n_own;
        for (int e = lane; e < n_own; e += 32) out[e] = acc[e];
        if (!OWN_V && CUT) {
            const double s = warp_sum(s_lane);
            if (lane == 0) part_s[slice * (a.batch * rows_own) + row] = s;
        }
    }
}

// ---- per row: slices added in order, then the split-frame gradient arithmetic once ---------------------------------
template <bool CUT>
__global__ void __launch_bounds__(TPB) sot_pairwise_rowgrad_kernel(const Args a, float* __restrict__ part_u,
                                                                   int slices_u, const double* __restrict__ part_s,
                                                                   float* __restrict__ part_v, int slices_v,
                                                                   float* __restrict__ grad_u,
                                                                   float* __restrict__ grad_v) {
    __shared__ double red[4 * NW];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const long long k = blockIdx.x, nu_rows = a.batch * a.rows_u, nv_rows = a.batch * a.rows_v;
    const RowPair rp{a.u + k * a.n, a.v + k * a.m, (grad_u != nullptr && k < nu_rows) ? a.n : 0,
                     (grad_v != nullptr && k < nv_rows) ? a.m : 0, (a.flags & FLAG_SQUARE) != 0};
    const int n = rp.n, m = rp.m, rows = n > m ? n : m, ntiles = (rows + TILE - 1) / TILE;
    const bool square = rp.square;
    float* const gu = part_u + k * a.n;  // slice 0 (the other slices follow at a stride of a whole slice)
    float* const gv = part_v + k * a.m;
    // my own entries of every tile: the slices added into slice 0 in order (no other thread reads them before)
    for (int t0 = 0; t0 < rows; t0 += TILE) {
        const int e0 = t0 + tid * E;
        for (int c = 0; c < E; ++c) {
            const int e = e0 + c;
            if (e < n) {
                float s = gu[e];
                for (int q = 1; q < slices_u; ++q) s += gu[q * nu_rows * a.n + e];
                gu[e] = s;
            }
            if (e < m) {
                float s = gv[e];
                for (int q = 1; q < slices_v; ++q) s += gv[q * nv_rows * a.m + e];
                gv[e] = s;
            }
        }
    }
    auto gpair = [&](int e) { return pack2(e < n ? gu[e] : 0.0f, e < m ? gv[e] : 0.0f); };
    const double mass_u = n > 0 ? a.mass_u[k] : 0.0, mass_v = m > 0 ? a.mass_v[k] : 0.0;
    Norm nm = normalise<false>(mass_u, mass_v, false);
    if (CUT) {  // v's 1/M_u was applied per pair; its mass has no derivative of its own
        nm.inv_v = 1.0;
        nm.v_live = false;
    }
    // ---- mass term: sum_i gw_i w_i = sum_t (S_t P_t + sum_i ls_i w_i), P_t = the CDF stage's prefix ----
    double dot_u = 0.0, dot_v = 0.0;
    if (nm.u_live || nm.v_live) {
        double car_u = 0.0, car_v = 0.0;
        for (int t0 = 0; t0 < rows; t0 += TILE) {
            f32x2 x2[E];
            load_tile(rp, t0, tid, x2);
            double ou_, ov_, nu = 0.0, nv = 0.0, tu, tv;
            tile_scan(rp, x2, ou_, ov_, nu, nv, tu, tv, red, tid);
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
        for (int q = 0; q < NW; ++q) {
            dot_u += red[2 * NW + q];
            dot_v += red[3 * NW + q];
        }
        __syncthreads();
        dot_u *= nm.inv_u;
        dot_v *= nm.inv_v;
    }
    if (CUT) {  // u's mass term also carries sum_j G_ij sum_l dL/dcv_l cv_l, summed by the sweep
        dot_v = 0.0;
        for (int q = 0; q < slices_u && n > 0; ++q) dot_v += part_s[q * nu_rows + k];
    }
    double corr_u, corr_v;
    mass_terms(nm, CUT, dot_u, dot_v, corr_u, corr_v);
    float ku, kv;
    grad_scale(nm, 1.0f, square, true, ku, kv);
    const f32x2 k2 = pack2(ku, kv);
    float* const ou = grad_u + k * a.n;
    float* const ov = grad_v + k * a.m;
    // ---- tiles in reverse: suffix sums of dL/dCDF, chain rule, x 2x ----
    double suf_u = 0.0, suf_v = 0.0;
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
            if (square) o2 = mul2(o2, pack2(e < n ? __ldg(rp.xu + e) : 0.0f, e < m ? __ldg(rp.xv + e) : 0.0f));
            float ga, gb;
            unpack2(o2, ga, gb);
            if (e < n) ou[e] = ga;
            if (e < m) ov[e] = gb;
        }
    }
}

// ---- exact k nearest v rows of every u row, with walks pruned by a quantile lower bound (DESIGN.md §4) -------------
// Q(t) = pos[min(lb(t), n - 1)] is the step quantile function of a stored CDF row (lb(t): entries below t); the walk
// integrates |Q_u - Q_v|^p over [0, max(end_u, end_v)].  a_l = the mean of Q over I_l = [l h, (l + 1) h], h = t0 / L,
// and Jensen on each interval gives D >= LB = h sum_l |a_u,l - a_v,l|^p.  The kernels compute LB from fp64 means and
// a pair is skipped only when LB (1 - eta) - eps exceeds tau, the k-th value walked so far: its fp32 value would then
// be strictly above tau (eta, eps and the shrink `del` of the means are derived in DESIGN.md §4).
constexpr int KL = 32;                      // intervals of [0, t0]
constexpr double kT0 = 1.0 - 0x1p-20;       // the bound covers [0, t0]; a row is bounded when its CDF ends >= t0
constexpr int KQ = 32;                      // queries (u rows) per CTA: one per lane
constexpr int KD = 32;                      // database (v) rows per tile: four per warp
constexpr int KW = 8;                       // warps per CTA
constexpr int kKnnCap = 128;                // largest k: the per-query lists are KQ * k (value, index) pairs in smem
constexpr int kMaxSlices = 256;             // database slices per query tile (merge heads per warp in smem)
constexpr long long kKnnTargetCtas = 592;   // CTAs the database is sliced for (4 per SM) ...
constexpr long long kMinSliceRows = 1024;   // ... in slices long enough for the threshold to tighten after its seeding

// The skip rule of both searches: LB = coef * S^expo (S = sum_l d_l, or sum_l d_l^2 when `squares`, expo = p / 2), and
// a pair of bounded rows is skipped when LB (1 - eta) - eps exceeds the threshold (bound_of below sets them).
struct Bound {
    double coef, expo, eta, eps;
    bool squares;
};

struct Knn {
    int k, slices;
    const double* emb_u;  // [batch * rows_u][KL] interval means, fp64
    const double* del_u;  // [batch * rows_u]: bound on their rounding, < 0 for a row without a bound
    const double* emb_v;
    const double* del_v;
    unsigned* tau;        // [batch * rows_u]: float bits of the smallest published k-th value (0xffffffff: none)
    float* lv;            // [batch * rows_u][slices][k]: each slice's sorted best values ...
    int* li;              // ... and their v row indices
    unsigned long long* walked;  // nullable
    Bound bd;
};

// total order of the results: value ascending, NaN after every number, then the lower index
SOT_DEVINL bool knn_less(float v, int i, float w, int j) {
    const bool nv = v != v, nw = w != w;
    if (nv != nw) return nw;
    if (!nv && v != w) return v < w;
    return i < j;
}

// One warp per row (u rows first, then v rows): lane l forms the mean of Q over I_l in fp64 and a bound on its rounding.
__global__ void __launch_bounds__(256) sot_pairwise_knn_embed_kernel(const Args a, double* __restrict__ emb_u,
                                                                    double* __restrict__ del_u,
                                                                    double* __restrict__ emb_v,
                                                                    double* __restrict__ del_v) {
    const int lane = threadIdx.x & 31;
    const long long row = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const long long nu_rows = a.batch * a.rows_u;
    if (row >= nu_rows + a.batch * a.rows_v) return;
    const bool is_u = row < nu_rows;
    const long long k = is_u ? row : row - nu_rows;
    const int n = is_u ? a.n : a.m;
    const float* const c = is_u ? a.cu + k * pad4(a.n + 2) : a.cv + k * pad4(a.m + 2);
    const float* const pos = is_u ? a.pos_u : a.pos_v;
    const double mass = is_u ? a.mass_u[k] : a.mass_v[k];
    // the walk integrates Q only for a non-decreasing row (NaN fails the test)
    bool ok = true;
    for (int i = lane; i < n; i += 32) ok = ok && c[i] >= (i > 0 ? c[i - 1] : 0.0f);
    const double h = kT0 / KL, lo = lane * h, hi = lo + h;  // (exact: t0 has 20 significant bits)
    int i = 0, top = n;  // first entry above lo: segment i is (c[i - 1], c[i]] (c[-1] = 0), where Q = pos[i]
    while (i < top) {
        const int mid = (i + top) >> 1;
        if (static_cast<double>(c[mid]) <= lo) i = mid + 1; else top = mid;
    }
    double sum = 0.0, asum = 0.0;
    for (; i < n; ++i) {
        const double s0 = fmax(i > 0 ? static_cast<double>(c[i - 1]) : 0.0, lo);
        const double s1 = fmin(static_cast<double>(c[i]), hi);
        if (s1 > s0) {
            const double x = pos[i];
            sum += x * (s1 - s0);
            asum += fabs(x) * (s1 - s0);
        }
        if (static_cast<double>(c[i]) >= hi) break;
    }
    const double mean = sum / h;
    // |fl(mean) - mean| <= (segments + 3) 2^-53 mean(|pos|) with at most n + 1 segments: twice that, for margin
    double del = static_cast<double>(n + 8) * 0x1p-52 * (asum / h);
    ok = ok && isfinite(mean) && isfinite(del);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) del = fmax(del, __shfl_xor_sync(FULL_MASK, del, off));
    const bool bounded = __all_sync(FULL_MASK, ok) && isfinite(mass) && static_cast<float>(mass) > SAFE_EPS &&
                         static_cast<double>(c[n - 1]) >= kT0;
    (is_u ? emb_u : emb_v)[k * KL + lane] = mean;
    if (lane == 0) (is_u ? del_u : del_v)[k] = bounded ? del : -1.0;
}

// The bounds of one tile of KQ queries x KD v rows: lane = query, warp w takes v rows w, w + 8, w + 16, w + 24 (the
// query means in shared memory [l][q], the v rows' means [j][l]).  keep[r] is cleared for a pair of bounded rows
// whose LB (1 - eta) - eps exceeds tau.  (sot_pairwise_knn_kernel has these lines inline: calling this helper there
// changes its instruction schedule.)
SOT_DEVINL void tile_bounds(const Bound& bd, const double* qemb, const double* qdel, const double* demb,
                            const double* ddel, int lane, int wid, double tau, bool (&keep)[KD / KW]) {
    constexpr int RPW = KD / KW;
    double s[RPW], shrink[RPW];
#pragma unroll
    for (int r = 0; r < RPW; ++r) {
        s[r] = 0.0;
        shrink[r] = qdel[lane] + ddel[wid + KW * r];
    }
#pragma unroll 8
    for (int l = 0; l < KL; ++l) {
        const double qa = qemb[l * KQ + lane];
#pragma unroll
        for (int r = 0; r < RPW; ++r) {
            const double d = fmax(fabs(qa - demb[(wid + KW * r) * KL + l]) - shrink[r], 0.0);
            s[r] = bd.squares ? fma(d, d, s[r]) : s[r] + d;
        }
    }
#pragma unroll
    for (int r = 0; r < RPW; ++r) {
        if (!keep[r] || qdel[lane] < 0.0 || ddel[wid + KW * r] < 0.0) continue;
        const double lb = bd.coef * (bd.expo == 1.0 ? s[r] : pow(s[r], bd.expo));
        keep[r] = !(lb * (1.0 - bd.eta) - bd.eps > tau);
    }
}

// One CTA per (batch entry, tile of KQ u rows, slice of the v rows).  Per tile of KD v rows: LB of the KQ x KD pairs
// against each query's threshold, the survivors walked one warp per pair on the CDF rows in global memory (walk_pair +
// warp_sum: the bits of sot_pairwise_loss_kernel), and each query's k best kept in shared memory.  The threshold is
// the smaller of this CTA's k-th value and the one other slices published with atomicMin.  PRUNE off (cut mode, the
// `qs > 1` mask): every pair is walked.  Writes the slice's sorted list of each query.
template <bool PRUNE, bool CUT>
__global__ void __launch_bounds__(256) sot_pairwise_knn_kernel(const Args a, const Knn kx) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int n = a.n, m = a.m, K = kx.k;
    double* const qemb = reinterpret_cast<double*>(smem);  // [KL][KQ]
    double* const qdel = qemb + KL * KQ;
    double* const demb = qdel + KQ;  // [KD][KL]
    double* const ddel = demb + KD * KL;
    float* const spu = reinterpret_cast<float*>(ddel + KD);
    float* const spv = spu + pad4(n);
    float* const lv = spv + pad4(m);  // [KQ][K]
    int* const li = reinterpret_cast<int*>(lv + KQ * K);
    int* const surv = li + KQ * K;  // [KQ * KD] survivors q * KD + j
    float* const sval = reinterpret_cast<float*>(surv + KQ * KD);
    float* const teff = sval + KQ * KD;  // [KQ] threshold of the tile
    float* const tloc = teff + KQ;       // [KQ] this CTA's k-th value (+inf until k numbers are kept)
    int* const lcnt = reinterpret_cast<int*>(tloc + KQ);
    int* const lworst = lcnt + KQ;
    int* const nsurv = lworst + KQ;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    long long blk = blockIdx.x;
    const int slice = static_cast<int>(blk % kx.slices);
    blk /= kx.slices;
    const long long qtiles = (a.rows_u + KQ - 1) / KQ;
    const long long qt = blk % qtiles, b = blk / qtiles;
    const int cnt_q = static_cast<int>(min(static_cast<long long>(KQ), a.rows_u - qt * KQ));
    const long long gq0 = b * a.rows_u + qt * KQ;  // global u row of query 0
    const long long lo = a.rows_v * slice / kx.slices, hi = a.rows_v * (slice + 1) / kx.slices;
    for (int e = tid; e < n; e += blockDim.x) spu[e] = a.pos_u[e];
    for (int e = tid; e < m; e += blockDim.x) spv[e] = a.pos_v[e];
    if constexpr (PRUNE) {
        for (int e = tid; e < KL * KQ; e += blockDim.x) {
            const int q = e % KQ, l = e / KQ;
            qemb[e] = q < cnt_q ? kx.emb_u[(gq0 + q) * KL + l] : 0.0;
        }
        if (tid < KQ) qdel[tid] = tid < cnt_q ? kx.del_u[gq0 + tid] : -1.0;
    }
    if (tid < KQ) {
        lcnt[tid] = 0;
        lworst[tid] = 0;
        tloc[tid] = f_inf();
    }
    const float thr = thr_of(a.flags);
    unsigned long long walked = 0;
    for (long long j0 = lo; j0 < hi; j0 += KD) {
        const int cnt_d = static_cast<int>(min(static_cast<long long>(KD), hi - j0));
        const long long gv0 = b * a.rows_v + j0;
        if constexpr (PRUNE) {
            for (int e = tid; e < KD * KL; e += blockDim.x)
                demb[e] = e / KL < cnt_d ? kx.emb_v[gv0 * KL + e] : 0.0;
            if (tid < KD) ddel[tid] = tid < cnt_d ? kx.del_v[gv0 + tid] : -1.0;
            if (tid < cnt_q) teff[tid] = fminf(tloc[tid], __uint_as_float(__ldcg(kx.tau + gq0 + tid)));  // (NaN: none)
        }
        if (tid == 0) *nsurv = 0;
        __syncthreads();
        // ---- bounds: lane = query, warp w takes v rows w, w + 8, w + 16, w + 24 of the tile ----
        {
            constexpr int RPW = KD / KW;
            bool keep[RPW];
#pragma unroll
            for (int r = 0; r < RPW; ++r) keep[r] = lane < cnt_q && wid + KW * r < cnt_d;
            if constexpr (PRUNE) {
                double s[RPW], shrink[RPW];
#pragma unroll
                for (int r = 0; r < RPW; ++r) {
                    s[r] = 0.0;
                    shrink[r] = qdel[lane] + ddel[wid + KW * r];
                }
#pragma unroll 8
                for (int l = 0; l < KL; ++l) {
                    const double qa = qemb[l * KQ + lane];
#pragma unroll
                    for (int r = 0; r < RPW; ++r) {
                        const double d = fmax(fabs(qa - demb[(wid + KW * r) * KL + l]) - shrink[r], 0.0);
                        s[r] = kx.bd.squares ? fma(d, d, s[r]) : s[r] + d;
                    }
                }
                const double tau = static_cast<double>(teff[lane]);
#pragma unroll
                for (int r = 0; r < RPW; ++r) {
                    if (!keep[r] || qdel[lane] < 0.0 || ddel[wid + KW * r] < 0.0) continue;
                    const double lb = kx.bd.coef * (kx.bd.expo == 1.0 ? s[r] : pow(s[r], kx.bd.expo));
                    keep[r] = !(lb * (1.0 - kx.bd.eta) - kx.bd.eps > tau);
                }
            }
#pragma unroll
            for (int r = 0; r < RPW; ++r)
                if (keep[r]) surv[atomicAdd(nsurv, 1)] = lane * KD + wid + KW * r;
        }
        __syncthreads();
        const int ns = *nsurv;
        walked += ns;
        // ---- walks: one warp per surviving pair ----
        for (int t = wid; t < ns; t += KW) {
            const int q = surv[t] / KD, j = surv[t] % KD;
            const long long gu = gq0 + q, gv = gv0 + j;
            const float* const crow_u = a.cu + gu * pad4(n + 2);
            const float* const crow_v = a.cv + gv * pad4(m + 2);
            VScale r;
            const double mu = a.mass_u[gu], mv = a.mass_v[gv];
            const Norm nm = pair_norm<CUT>(mu, mv, crow_v, m, r);
            const bool finite = finite_frame(mu, mv, nm);  // (warp uniform)
            float acc = 0.0f;
            if (finite)
                acc = walk_pair<false, CUT>(PairRows{crow_u, crow_v, spu, spv, n, m, r, a.p, thr}, lane, nullptr,
                                            [](int, float) {});
            const double s = warp_sum(static_cast<double>(acc));
            if (lane == 0) sval[t] = finite ? static_cast<float>(s) : f_nan();
        }
        __syncthreads();
        // ---- each query's thread keeps its k best ----
        if (tid < cnt_q) {
            float* const L = lv + tid * K;
            int* const I = li + tid * K;
            int cnt = lcnt[tid], worst = lworst[tid];
            const auto find_worst = [&]() {
                worst = 0;
                for (int e = 1; e < K; ++e)
                    if (knn_less(L[worst], I[worst], L[e], I[e])) worst = e;
            };
            for (int t = 0; t < ns; ++t) {
                if (surv[t] / KD != tid) continue;
                const float v = sval[t];
                const int idx = static_cast<int>(j0) + surv[t] % KD;
                if (cnt < K) {
                    L[cnt] = v;
                    I[cnt] = idx;
                    if (++cnt == K) find_worst();
                } else if (knn_less(v, idx, L[worst], I[worst])) {
                    L[worst] = v;
                    I[worst] = idx;
                    find_worst();
                }
            }
            lcnt[tid] = cnt;
            lworst[tid] = worst;
            // publish the k-th value: a number walked here, never NaN (and +0 for a -0)
            if (PRUNE && cnt == K && L[worst] == L[worst] && L[worst] < tloc[tid]) {
                tloc[tid] = L[worst];
                atomicMin(kx.tau + gq0 + tid, __float_as_uint(L[worst] + 0.0f));
            }
        }
        __syncthreads();
    }
    // ---- the slice's list of each query, sorted; empty places hold (NaN, INT_MAX), which rank last ----
    if (tid < cnt_q) {
        float* const L = lv + tid * K;
        int* const I = li + tid * K;
        const int cnt = lcnt[tid];
        for (int e = 1; e < cnt; ++e) {
            const float v = L[e];
            const int idx = I[e];
            int f = e;
            for (; f > 0 && knn_less(v, idx, L[f - 1], I[f - 1]); --f) {
                L[f] = L[f - 1];
                I[f] = I[f - 1];
            }
            L[f] = v;
            I[f] = idx;
        }
        const long long at = ((gq0 + tid) * kx.slices + slice) * K;
        for (int e = 0; e < K; ++e) {
            kx.lv[at + e] = e < cnt ? L[e] : f_nan();
            kx.li[at + e] = e < cnt ? I[e] : 0x7fffffff;
        }
    }
    if (tid == 0 && kx.walked != nullptr) atomicAdd(kx.walked, walked);
}

// One warp per query: the k smallest of its slices' sorted lists, in order.
__global__ void __launch_bounds__(256) sot_pairwise_knn_merge_kernel(const Knn kx, long long queries,
                                                                    float* __restrict__ values,
                                                                    int64_t* __restrict__ indices) {
    __shared__ int head[KW][kMaxSlices];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long q = static_cast<long long>(blockIdx.x) * KW + wid;
    if (q >= queries) return;
    const int S = kx.slices, K = kx.k;
    for (int s = lane; s < S; s += 32) head[wid][s] = 0;
    __syncwarp();
    const long long base = q * S * K;
    for (int e = 0; e < K; ++e) {
        float bv = f_nan();
        int bi = 0x7fffffff, bs = 0x7fffffff;
        for (int s = lane; s < S; s += 32) {
            const int h = head[wid][s];
            if (h >= K) continue;
            const float v = kx.lv[base + s * K + h];
            const int i = kx.li[base + s * K + h];
            if (knn_less(v, i, bv, bi) || (!knn_less(bv, bi, v, i) && s < bs)) {
                bv = v;
                bi = i;
                bs = s;
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const float v = __shfl_xor_sync(FULL_MASK, bv, off);
            const int i = __shfl_xor_sync(FULL_MASK, bi, off), s = __shfl_xor_sync(FULL_MASK, bs, off);
            if (knn_less(v, i, bv, bi) || (!knn_less(bv, bi, v, i) && s < bs)) {
                bv = v;
                bi = i;
                bs = s;
            }
        }
        if (lane == 0) {
            values[q * K + e] = bv;
            indices[q * K + e] = bi;
            head[wid][bs] += 1;
        }
        __syncwarp();
    }
}

// ---- every v row within a fixed radius of each u row, with the same bound and walk (DESIGN.md §4) -----------------
constexpr long long kRadiusTargetCtas = 4736;    // CTAs the database is sliced for (about ten waves of three per SM,
constexpr long long kRadiusMinSliceRows = 1024;  // so that uneven hit counts even out); slices need no merge step

struct Radius {
    int slices;
    float radius;
    long long capacity;
    const double* emb_u;  // as in Knn
    const double* del_u;
    const double* emb_v;
    const double* del_v;
    unsigned long long* count;   // pairs within the radius
    unsigned long long* keys;    // [capacity]: (b P + i) R + j of each of them, in no particular order ...
    float* vals;                 // ... and its distance
    unsigned long long* walked;  // nullable
    Bound bd;
};

// One CTA per (batch entry, tile of KQ u rows, slice of the v rows), as in sot_pairwise_knn_kernel, with the radius
// as every query's threshold from the first tile on.  Per tile of KD v rows: the bounds, the survivors walked one warp
// per pair (walk_pair + warp_sum: the bits of sot_pairwise_loss_kernel), and the pairs with dist <= radius reserved
// slots with one atomicAdd on the counter per tile; slots at or past `capacity` are counted but not written.  PRUNE
// off (cut mode, the `qs > 1` mask): every pair is walked.
template <bool PRUNE, bool CUT>
__global__ void __launch_bounds__(256) sot_pairwise_radius_kernel(const Args a, const Radius rx) {
    extern __shared__ __align__(16) unsigned char smem[];
    const int n = a.n, m = a.m;
    double* const qemb = reinterpret_cast<double*>(smem);  // [KL][KQ]
    double* const qdel = qemb + KL * KQ;
    double* const demb = qdel + KQ;  // [KD][KL]
    double* const ddel = demb + KD * KL;
    float* const spu = reinterpret_cast<float*>(ddel + KD);
    float* const spv = spu + pad4(n);
    int* const surv = reinterpret_cast<int*>(spv + pad4(m));  // [KQ * KD] survivors q * KD + j
    int* const hit = surv + KQ * KD;                         // [KQ * KD] the survivors within the radius ...
    float* const hval = reinterpret_cast<float*>(hit + KQ * KD);  // ... and their distances
    unsigned long long* const hbase = reinterpret_cast<unsigned long long*>(hval + KQ * KD);  // the tile's first slot
    int* const nsurv = reinterpret_cast<int*>(hbase + 1);
    int* const nhit = nsurv + 1;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    long long blk = blockIdx.x;
    const int slice = static_cast<int>(blk % rx.slices);
    blk /= rx.slices;
    const long long qtiles = (a.rows_u + KQ - 1) / KQ;
    const long long qt = blk % qtiles, b = blk / qtiles;
    const int cnt_q = static_cast<int>(min(static_cast<long long>(KQ), a.rows_u - qt * KQ));
    const long long gq0 = b * a.rows_u + qt * KQ;  // global u row of query 0, b P + i
    const long long lo = a.rows_v * slice / rx.slices, hi = a.rows_v * (slice + 1) / rx.slices;
    for (int e = tid; e < n; e += blockDim.x) spu[e] = a.pos_u[e];
    for (int e = tid; e < m; e += blockDim.x) spv[e] = a.pos_v[e];
    if constexpr (PRUNE) {
        for (int e = tid; e < KL * KQ; e += blockDim.x) {
            const int q = e % KQ, l = e / KQ;
            qemb[e] = q < cnt_q ? rx.emb_u[(gq0 + q) * KL + l] : 0.0;
        }
        if (tid < KQ) qdel[tid] = tid < cnt_q ? rx.del_u[gq0 + tid] : -1.0;
    }
    const float thr = thr_of(a.flags), radius = rx.radius;
    unsigned long long walked = 0;
    for (long long j0 = lo; j0 < hi; j0 += KD) {
        const int cnt_d = static_cast<int>(min(static_cast<long long>(KD), hi - j0));
        const long long gv0 = b * a.rows_v + j0;
        if constexpr (PRUNE) {
            for (int e = tid; e < KD * KL; e += blockDim.x)
                demb[e] = e / KL < cnt_d ? rx.emb_v[gv0 * KL + e] : 0.0;
            if (tid < KD) ddel[tid] = tid < cnt_d ? rx.del_v[gv0 + tid] : -1.0;
        }
        if (tid == 0) {
            *nsurv = 0;
            *nhit = 0;
        }
        __syncthreads();
        {
            bool keep[KD / KW];
#pragma unroll
            for (int r = 0; r < KD / KW; ++r) keep[r] = lane < cnt_q && wid + KW * r < cnt_d;
            if constexpr (PRUNE) tile_bounds(rx.bd, qemb, qdel, demb, ddel, lane, wid, radius, keep);
#pragma unroll
            for (int r = 0; r < KD / KW; ++r)
                if (keep[r]) surv[atomicAdd(nsurv, 1)] = lane * KD + wid + KW * r;
        }
        __syncthreads();
        const int ns = *nsurv;
        walked += ns;
        for (int t = wid; t < ns; t += KW) {
            const int q = surv[t] / KD, j = surv[t] % KD;
            const long long gu = gq0 + q, gv = gv0 + j;
            const float* const crow_u = a.cu + gu * pad4(n + 2);
            const float* const crow_v = a.cv + gv * pad4(m + 2);
            VScale r;
            const double mu = a.mass_u[gu], mv = a.mass_v[gv];
            const Norm nm = pair_norm<CUT>(mu, mv, crow_v, m, r);
            const bool finite = finite_frame(mu, mv, nm);  // (warp uniform)
            float acc = 0.0f;
            if (finite)
                acc = walk_pair<false, CUT>(PairRows{crow_u, crow_v, spu, spv, n, m, r, a.p, thr}, lane, nullptr,
                                            [](int, float) {});
            const double s = warp_sum(static_cast<double>(acc));
            const float d = finite ? static_cast<float>(s) : f_nan();
            if (lane == 0 && d <= radius) {  // (NaN never counts)
                const int h = atomicAdd(nhit, 1);
                hit[h] = surv[t];
                hval[h] = d;
            }
        }
        __syncthreads();
        const int nh = *nhit;
        if (nh > 0) {  // (CTA uniform)
            if (tid == 0) *hbase = atomicAdd(rx.count, static_cast<unsigned long long>(nh));
            __syncthreads();
            const unsigned long long at = *hbase;
            for (int e = tid; e < nh; e += blockDim.x) {
                if (at + e >= static_cast<unsigned long long>(rx.capacity)) break;
                const int q = hit[e] / KD, j = hit[e] % KD;
                rx.keys[at + e] = static_cast<unsigned long long>((gq0 + q) * a.rows_v + j0 + j);
                rx.vals[at + e] = hval[e];
            }
        }
        __syncthreads();  // the tile's lists and counters are reused by the next one
    }
    if (tid == 0 && rx.walked != nullptr) atomicAdd(rx.walked, walked);
}

// The keys, sorted into `rows`, split in place into the row b P + i and the column j of each of the first
// min(count, capacity) pairs.
__global__ void __launch_bounds__(256) sot_pairwise_radius_split_kernel(const unsigned long long* __restrict__ count,
                                                                       long long capacity, long long rows_v,
                                                                       int64_t* __restrict__ rows,
                                                                       int64_t* __restrict__ cols) {
    const long long e = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (e >= capacity || static_cast<unsigned long long>(e) >= *count) return;
    const long long key = rows[e], row = key / rows_v;
    rows[e] = row;
    cols[e] = key - row * rows_v;
}

// ---- host side ------------------------------------------------------------------------------------------------------
// Largest tile (rows of each side) whose shared memory fits the budget; 1 otherwise (<= 169 KB at 8448 bins).
int tile_rows(int n, int m, bool grad) {
    for (int t = 8; t > 1; t >>= 1) {
        long long bytes = 4 * (pad4(n) + pad4(m)) + 4LL * t * (pad4(n + 2) + pad4(m + 2)) + 16;
        bytes += grad ? 4LL * t * (pad4(n > m ? n : m) + 32) : 4LL * 32 * 8;
        if (bytes <= kSmemBudget) return t;
    }
    return 1;
}

long long smem_bytes(const Args& a, bool grad, bool own_v) {
    const int T = a.tile;
    long long bytes = 4 * (pad4(a.n) + pad4(a.m)) + 4LL * T * (pad4(a.n + 2) + pad4(a.m + 2)) + 16;
    return bytes + (grad ? 4LL * T * (pad4(own_v ? a.m : a.n) + 32) : 4LL * 32 * 8);
}

template <auto kernel>
cudaError_t allow_smem() {
    static std::atomic<bool> done[64];  // per kernel (template argument) and device ordinal
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev >= 0 && dev < 64 && done[dev].load(std::memory_order_acquire)) return cudaSuccess;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e == cudaSuccess && dev >= 0 && dev < 64) done[dev].store(true, std::memory_order_release);
    return e;
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

// The constants of the skip rule for p and rows of n and m bins (DESIGN.md §4).
Bound bound_of(float p, int n, int m) {
    Bound bd{};
    // LB = h sum_l d_l^p >= h L^(1 - e) (sum_l d_l^(p / e))^e with e = p / 2 for p >= 2 (sums of squares), else e = p
    const double pd = p, h = kT0 / KL;
    bd.squares = pd >= 2.0;
    bd.expo = bd.squares ? pd / 2.0 : pd;
    bd.coef = h * std::pow(static_cast<double>(KL), 1.0 - bd.expo);
    // relative rounding of the fp32 walk (lane sums of ceil((n + m) / 32) terms, the step, the gap, |d|^p, the sum and
    // the cast) and of the fp64 bound; eps: absolute error of subnormal terms
    const long long per_lane = (n + m + 31) / 32;
    bd.eta = (static_cast<double>(per_lane) + std::ceil(pd) + 16.0) * 0x1p-24 + (pd + 1.0) * 0x1p-40;
    bd.eps = 0x1p-100;
    return bd;
}

}  // namespace pairwise
}  // namespace sot

namespace {

using sot::fail;
using sot::pairwise::Args;
using sot::pairwise::pad4;

// sizes, flags, p and bins: the rules every pairwise entry point shares
int validate_rows(const sot_pairwise_problem* p) {
    if (p == nullptr) return fail(SOT_EINVAL, "problem is NULL");
    if (p->batch < 0 || p->rows_u < 0 || p->rows_v < 0 || p->n_u < 1 || p->n_v < 1)
        return fail(SOT_EINVAL, "bad sizes: batch=%lld rows_u=%lld rows_v=%lld n_u=%d n_v=%d", (long long)p->batch,
                    (long long)p->rows_u, (long long)p->rows_v, p->n_u, p->n_v);
    if (p->flags & (SOT_RAW_WEIGHTS | SOT_COMPLEX_INPUT | SOT_UNIFORM_GRID))
        return fail(SOT_EINVAL, "pairwise distances take SOT_SQUARE, SOT_CUT_SCALE and SOT_LIMIT only (raw weights and "
                    "complex rows are not supported)");
    if (p->flags & ~(SOT_SQUARE | SOT_CUT_SCALE | SOT_LIMIT)) return fail(SOT_EINVAL, "unknown flag bits");
    if (!(p->p >= 1.0f)) return fail(SOT_EDOMAIN, "The OT loss is only valid for p>=1, %g was given", (double)p->p);
    if (p->n_u > sot::pairwise::kMaxBins || p->n_v > sot::pairwise::kMaxBins)
        return fail(SOT_ETOOBIG, "pairwise rows of %d / %d bins: the limit is %d bins", p->n_u, p->n_v,
                    sot::pairwise::kMaxBins);
    return SOT_OK;
}

int validate_pairwise(const sot_pairwise_problem* p) {
    if (int rc = validate_rows(p)) return rc;
    // every grid (one CTA per row index, per tile of T x T pairs, at worst T = 1) within 2^31 - 1 CTAs
    const long long rows = p->rows_u > p->rows_v ? p->rows_u : p->rows_v;
    if (p->batch > 0 && rows > 0 && (p->rows_u > 0x7fffffffLL / p->batch / (p->rows_v > 0 ? p->rows_v : 1) ||
                                     rows > 0x7fffffffLL / p->batch))
        return fail(SOT_ETOOBIG, "too many pairs for one launch (batch x rows_u x rows_v above 2^31 - 1)");
    if (p->batch * p->rows_u * p->rows_v == 0) return SOT_OK;
    if (p->u == nullptr || p->v == nullptr || p->pos_u == nullptr || p->pos_v == nullptr)
        return fail(SOT_EINVAL, "u, v, pos_u or pos_v is NULL");
    return SOT_OK;
}

Args args_of(const sot_pairwise_problem* p) {
    Args a{};
    a.batch = p->batch;
    a.rows_u = p->rows_u;
    a.rows_v = p->rows_v;
    a.n = p->n_u;
    a.m = p->n_v;
    a.u = p->u;
    a.v = p->v;
    a.pos_u = p->pos_u;
    a.pos_v = p->pos_v;
    a.p = p->p;
    a.flags = p->flags;
    return a;
}

// CDF and mass scratch of the pre-pass, carved from `c`; the pointers are filled in once the block exists
struct CdfScratch {
    long long cu, cv, mu, mv;
};
CdfScratch carve_cdfs(sot::pairwise::Carve& c, const Args& a) {
    return {c.take(4 * a.batch * a.rows_u * pad4(a.n + 2)), c.take(4 * a.batch * a.rows_v * pad4(a.m + 2)),
            c.take(8 * a.batch * a.rows_u), c.take(8 * a.batch * a.rows_v)};
}
void place_cdfs(Args& a, const CdfScratch& s, char* base) {
    a.cu = reinterpret_cast<float*>(base + s.cu);
    a.cv = reinterpret_cast<float*>(base + s.cv);
    a.mass_u = reinterpret_cast<double*>(base + s.mu);
    a.mass_v = reinterpret_cast<double*>(base + s.mv);
}

int launch_cdfs(const Args& a, cudaStream_t stream) {
    const long long rows = a.batch * (a.rows_u > a.rows_v ? a.rows_u : a.rows_v);
    sot::pairwise::sot_pairwise_cdf_kernel<<<static_cast<unsigned>(rows), sot::pairwise::TPB, 0, stream>>>(a);
    return sot::launched(cudaGetLastError(), "sot_pairwise_cdf_kernel");
}

template <auto kernel, typename... Rest>
cudaError_t launch_big(long long grid, int threads, long long smem, cudaStream_t stream, Rest... rest) {
    const cudaError_t e = sot::pairwise::allow_smem<kernel>();
    if (e != cudaSuccess) return e;
    kernel<<<static_cast<unsigned>(grid), threads, static_cast<size_t>(smem), stream>>>(rest...);
    return cudaGetLastError();
}

// frees the scratch on the stream whatever happened before; the first error wins
int finish(int rc, void* scratch, cudaStream_t stream) {
    const cudaError_t e = cudaFreeAsync(scratch, stream);
    if (rc == SOT_OK && e != cudaSuccess) return fail(static_cast<int>(e), "cudaFreeAsync: %s", cudaGetErrorString(e));
    return rc;
}

// the interval means of every u and v row (after the CDF pre-pass): what both searches prune with
int launch_embed(const Args& a, double* emb_u, double* del_u, double* emb_v, double* del_v, cudaStream_t s) {
    using sot::pairwise::KW;
    const long long grid = (a.batch * (a.rows_u + a.rows_v) + KW - 1) / KW;
    sot::pairwise::sot_pairwise_knn_embed_kernel<<<static_cast<unsigned>(grid), 32 * KW, 0, s>>>(a, emb_u, del_u,
                                                                                                  emb_v, del_v);
    return sot::launched(cudaGetLastError(), "sot_pairwise_knn_embed_kernel");
}

// both searches cap B * P and B * R, not the pairs; the inputs are read when there is a pair (`any`)
int validate_search(const sot_pairwise_problem* p, bool any) {
    if (p->batch > 0 && (p->rows_u > 0x7fffffffLL / p->batch || p->rows_v > 0x7fffffffLL / p->batch))
        return fail(SOT_ETOOBIG, "too many rows for one launch (batch x rows above 2^31 - 1)");
    if (any && (p->u == nullptr || p->v == nullptr || p->pos_u == nullptr || p->pos_v == nullptr))
        return fail(SOT_EINVAL, "u, v, pos_u or pos_v is NULL");
    return SOT_OK;
}

}  // namespace

namespace sot {
namespace pairwise {

// `rows` unpaired rows of n bins as one pairwise problem: the first half is the u lane, the rest the v lane, so the
// lanes' CDF rows, masses, dL/dCDF rows and gradient rows each follow one another in the caller's buffers.
static Args unpaired(const float* x, long long rows, int n, bool square, float* cdf, double* mass) {
    const long long h = (rows + 1) / 2;
    Args a{};
    a.batch = 1;
    a.rows_u = h;
    a.rows_v = rows - h;
    a.n = a.m = n;
    a.u = x;
    a.v = x + h * n;
    a.flags = square ? FLAG_SQUARE : 0;
    a.cu = cdf;
    a.cv = cdf + h * pad4(n + 2);
    a.mass_u = mass;
    a.mass_v = mass + h;
    return a;
}

int launch_row_cdfs(const float* x, long long rows, int n, bool square, float* cdf, double* mass, cudaStream_t s) {
    return launch_cdfs(unpaired(x, rows, n, square, cdf, mass), s);
}

int launch_row_grads(const float* x, long long rows, int n, bool square, const double* mass, float* dcdf, float* grad,
                     cudaStream_t s) {
    const Args a = unpaired(x, rows, n, square, nullptr, const_cast<double*>(mass));
    const long long h = a.rows_u;
    sot_pairwise_rowgrad_kernel<false><<<static_cast<unsigned>(h), TPB, 0, s>>>(a, dcdf, 1, nullptr, dcdf + h * n, 1,
                                                                                  grad, grad + h * n);
    return sot::launched(cudaGetLastError(), "sot_pairwise_rowgrad_kernel");
}

}  // namespace pairwise
}  // namespace sot

extern "C" {

int sot_pairwise_device(const sot_pairwise_problem* prob, float* dist, void* stream) {
    if (int rc = validate_pairwise(prob)) return rc;
    if (prob->batch * prob->rows_u * prob->rows_v == 0) return SOT_OK;
    if (dist == nullptr) return fail(SOT_EINVAL, "dist is NULL");
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    Args a = args_of(prob);
    a.tile = sot::pairwise::tile_rows(a.n, a.m, false);
    sot::pairwise::Carve c;
    const CdfScratch cs = carve_cdfs(c, a);
    char* scratch = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&scratch), static_cast<size_t>(c.bytes), s);
    if (e != cudaSuccess) return fail(static_cast<int>(e), "pairwise scratch: %s", cudaGetErrorString(e));
    place_cdfs(a, cs, scratch);
    int rc = launch_cdfs(a, s);
    if (rc == SOT_OK) {
        const int T = a.tile;
        const long long grid = a.batch * ((a.rows_u + T - 1) / T) * ((a.rows_v + T - 1) / T);
        const int threads = 32 * (T * T < 8 ? T * T : 8);
        const long long smem = sot::pairwise::smem_bytes(a, false, false);
        e = (a.flags & SOT_CUT_SCALE)
                ? launch_big<sot::pairwise::sot_pairwise_loss_kernel<true>>(grid, threads, smem, s, a, dist)
                : launch_big<sot::pairwise::sot_pairwise_loss_kernel<false>>(grid, threads, smem, s, a, dist);
        rc = sot::launched(e, "sot_pairwise_loss_kernel");
    }
    return finish(rc, scratch, s);
}

int sot_pairwise_backward_device(const sot_pairwise_problem* prob, const float* upstream, float* grad_u,
                                 float* grad_v, void* stream) {
    if (int rc = validate_pairwise(prob)) return rc;
    if (prob->batch * prob->rows_u * prob->rows_v == 0 || (grad_u == nullptr && grad_v == nullptr)) return SOT_OK;
    if (upstream == nullptr) return fail(SOT_EINVAL, "upstream is NULL");
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    const bool cut = prob->flags & SOT_CUT_SCALE;
    Args a = args_of(prob);
    a.tile = sot::pairwise::tile_rows(a.n, a.m, true);
    const int T = a.tile;
    const long long tiles_u = (a.rows_u + T - 1) / T, tiles_v = (a.rows_v + T - 1) / T;
    // slices of the partner range: about kTargetCtas CTAs per batch entry, so that the summation order (and so every
    // bit of the gradients) does not depend on the batch size.  Scratch: min(slices) partial copies of the gradient
    // rows, at most ceil(kTargetCtas / tiles of the owned side) and at most the partner's tile count.
    auto slices_for = [&](long long tiles_own, long long tiles_str) {
        const long long q = (sot::pairwise::kTargetCtas + tiles_own - 1) / tiles_own;
        return static_cast<int>(q < tiles_str ? q : tiles_str);
    };
    const int slices_u = grad_u != nullptr ? slices_for(tiles_u, tiles_v) : 0;
    const int slices_v = grad_v != nullptr ? slices_for(tiles_v, tiles_u) : 0;
    sot::pairwise::Carve c;
    const CdfScratch cs = carve_cdfs(c, a);
    const long long at_pu = c.take(4LL * slices_u * a.batch * a.rows_u * a.n);
    const long long at_ps = c.take(8LL * (cut ? slices_u : 0) * a.batch * a.rows_u);
    const long long at_pv = c.take(4LL * slices_v * a.batch * a.rows_v * a.m);
    char* scratch = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&scratch), static_cast<size_t>(c.bytes), s);
    if (e != cudaSuccess) return fail(static_cast<int>(e), "pairwise scratch: %s", cudaGetErrorString(e));
    place_cdfs(a, cs, scratch);
    float* const part_u = reinterpret_cast<float*>(scratch + at_pu);
    double* const part_s = reinterpret_cast<double*>(scratch + at_ps);
    float* const part_v = reinterpret_cast<float*>(scratch + at_pv);
    int rc = launch_cdfs(a, s);
    using sot::pairwise::sot_pairwise_grad_kernel;
    if (rc == SOT_OK && grad_u != nullptr) {
        const long long grid = a.batch * tiles_u * slices_u, smem = sot::pairwise::smem_bytes(a, true, false);
        e = cut ? launch_big<sot_pairwise_grad_kernel<false, true>>(grid, 32 * T, smem, s, a, upstream, part_u, part_s,
                             slices_u)
                : launch_big<sot_pairwise_grad_kernel<false, false>>(grid, 32 * T, smem, s, a, upstream, part_u,
                             part_s, slices_u);
        rc = sot::launched(e, "sot_pairwise_grad_kernel");
    }
    if (rc == SOT_OK && grad_v != nullptr) {
        const long long grid = a.batch * tiles_v * slices_v, smem = sot::pairwise::smem_bytes(a, true, true);
        e = cut ? launch_big<sot_pairwise_grad_kernel<true, true>>(grid, 32 * T, smem, s, a, upstream, part_v, part_s,
                             slices_v)
                : launch_big<sot_pairwise_grad_kernel<true, false>>(grid, 32 * T, smem, s, a, upstream, part_v,
                             part_s, slices_v);
        rc = sot::launched(e, "sot_pairwise_grad_kernel");
    }
    if (rc == SOT_OK) {
        const long long grid = a.batch * (a.rows_u > a.rows_v ? a.rows_u : a.rows_v);
        const unsigned g = static_cast<unsigned>(grid);
        if (cut)
            sot::pairwise::sot_pairwise_rowgrad_kernel<true><<<g, sot::pairwise::TPB, 0, s>>>(
                a, part_u, slices_u, part_s, part_v, slices_v, grad_u, grad_v);
        else
            sot::pairwise::sot_pairwise_rowgrad_kernel<false><<<g, sot::pairwise::TPB, 0, s>>>(
                a, part_u, slices_u, part_s, part_v, slices_v, grad_u, grad_v);
        rc = sot::launched(cudaGetLastError(), "sot_pairwise_rowgrad_kernel");
    }
    return finish(rc, scratch, s);
}

int sot_pairwise_knn_device(const sot_pairwise_problem* prob, int32_t k, float* values, int64_t* indices,
                            int64_t* walked, void* stream) {
    using namespace sot::pairwise;
    if (int rc = validate_rows(prob)) return rc;
    if (k < 1 || k > kKnnCap || k > prob->rows_v)
        return fail(SOT_EINVAL, "k = %d: it must be at least 1 and at most min(rows_v = %lld, %d)", k,
                    (long long)prob->rows_v, kKnnCap);
    const long long BP = prob->batch * prob->rows_u, BR = prob->batch * prob->rows_v;
    if (int rc = validate_search(prob, BP > 0)) return rc;
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    if (BP > 0 && (values == nullptr || indices == nullptr)) return fail(SOT_EINVAL, "values or indices is NULL");
    if (walked != nullptr) {
        const cudaError_t e = cudaMemsetAsync(walked, 0, sizeof(int64_t), s);
        if (e != cudaSuccess) return fail(static_cast<int>(e), "cudaMemsetAsync: %s", cudaGetErrorString(e));
    }
    if (BP == 0) return SOT_OK;
    const bool cut = prob->flags & SOT_CUT_SCALE, prune = !(prob->flags & (SOT_CUT_SCALE | SOT_LIMIT));
    Args a = args_of(prob);
    const long long qtiles = (a.rows_u + KQ - 1) / KQ;
    const long long long_slices = (a.rows_v + kMinSliceRows - 1) / kMinSliceRows;
    long long S = (kKnnTargetCtas + a.batch * qtiles - 1) / (a.batch * qtiles);
    S = S < long_slices ? S : long_slices;
    S = S < kMaxSlices ? S : kMaxSlices;
    Knn kx{};
    kx.k = k;
    kx.slices = static_cast<int>(S);
    kx.walked = reinterpret_cast<unsigned long long*>(walked);
    kx.bd = bound_of(prob->p, a.n, a.m);
    sot::pairwise::Carve c;
    const CdfScratch cs = carve_cdfs(c, a);
    const long long at_eu = c.take(prune ? 8LL * KL * BP : 0), at_du = c.take(prune ? 8LL * BP : 0);
    const long long at_ev = c.take(prune ? 8LL * KL * BR : 0), at_dv = c.take(prune ? 8LL * BR : 0);
    const long long at_tau = c.take(4LL * BP);
    const long long at_lv = c.take(4LL * BP * S * k), at_li = c.take(4LL * BP * S * k);
    char* scratch = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&scratch), static_cast<size_t>(c.bytes), s);
    if (e != cudaSuccess) return fail(static_cast<int>(e), "pairwise scratch: %s", cudaGetErrorString(e));
    place_cdfs(a, cs, scratch);
    double* const emb_u = reinterpret_cast<double*>(scratch + at_eu);
    double* const del_u = reinterpret_cast<double*>(scratch + at_du);
    double* const emb_v = reinterpret_cast<double*>(scratch + at_ev);
    double* const del_v = reinterpret_cast<double*>(scratch + at_dv);
    kx.emb_u = emb_u;
    kx.del_u = del_u;
    kx.emb_v = emb_v;
    kx.del_v = del_v;
    kx.tau = reinterpret_cast<unsigned*>(scratch + at_tau);
    kx.lv = reinterpret_cast<float*>(scratch + at_lv);
    kx.li = reinterpret_cast<int*>(scratch + at_li);
    e = cudaMemsetAsync(kx.tau, 0xff, 4 * static_cast<size_t>(BP), s);  // no threshold published yet
    int rc = e == cudaSuccess ? SOT_OK : fail(static_cast<int>(e), "cudaMemsetAsync: %s", cudaGetErrorString(e));
    if (rc == SOT_OK) rc = launch_cdfs(a, s);
    if (rc == SOT_OK && prune) rc = launch_embed(a, emb_u, del_u, emb_v, del_v, s);
    if (rc == SOT_OK) {
        const long long grid = a.batch * qtiles * S;
        const long long smem = 8LL * (KL * KQ + KQ + KD * KL + KD) +
                               4LL * (pad4(a.n) + pad4(a.m) + 2LL * KQ * k + 2LL * KQ * KD + 4 * KQ + 1);
        e = prune ? launch_big<sot_pairwise_knn_kernel<true, false>>(grid, 32 * KW, smem, s, a, kx)
            : cut ? launch_big<sot_pairwise_knn_kernel<false, true>>(grid, 32 * KW, smem, s, a, kx)
                  : launch_big<sot_pairwise_knn_kernel<false, false>>(grid, 32 * KW, smem, s, a, kx);
        rc = sot::launched(e, "sot_pairwise_knn_kernel");
    }
    if (rc == SOT_OK) {
        sot_pairwise_knn_merge_kernel<<<static_cast<unsigned>((BP + KW - 1) / KW), 32 * KW, 0, s>>>(kx, BP, values,
                                                                                                   indices);
        rc = sot::launched(cudaGetLastError(), "sot_pairwise_knn_merge_kernel");
    }
    return finish(rc, scratch, s);
}

int sot_pairwise_radius_device(const sot_pairwise_problem* prob, float radius, int64_t capacity, int64_t* rows,
                               int64_t* cols, float* values, int64_t* count, int64_t* walked, void* stream) {
    using namespace sot::pairwise;
    if (int rc = validate_rows(prob)) return rc;
    if (radius != radius) return fail(SOT_EINVAL, "the radius is NaN");
    if (capacity < 0) return fail(SOT_EINVAL, "capacity = %lld: it must be at least 0", (long long)capacity);
    const long long BP = prob->batch * prob->rows_u, BR = prob->batch * prob->rows_v;
    const long long pairs = BP * prob->rows_v;  // (< 2^62 under the caps)
    if (int rc = validate_search(prob, pairs > 0)) return rc;
    if (count == nullptr) return fail(SOT_EINVAL, "count is NULL");
    if (pairs > 0 && capacity > 0 && (rows == nullptr || cols == nullptr || values == nullptr))
        return fail(SOT_EINVAL, "rows, cols or values is NULL");
    const cudaStream_t s = static_cast<cudaStream_t>(stream);
    for (int64_t* counter : {count, walked}) {
        if (counter == nullptr) continue;
        const cudaError_t e = cudaMemsetAsync(counter, 0, sizeof(int64_t), s);
        if (e != cudaSuccess) return fail(static_cast<int>(e), "cudaMemsetAsync: %s", cudaGetErrorString(e));
    }
    if (pairs == 0) return SOT_OK;
    const bool cut = prob->flags & SOT_CUT_SCALE, prune = !(prob->flags & (SOT_CUT_SCALE | SOT_LIMIT));
    const long long cap = capacity < pairs ? capacity : pairs;  // (no more slots can be used)
    Args a = args_of(prob);
    const long long qtiles = (a.rows_u + KQ - 1) / KQ;
    const long long long_slices = (a.rows_v + kRadiusMinSliceRows - 1) / kRadiusMinSliceRows;
    long long S = (kRadiusTargetCtas + a.batch * qtiles - 1) / (a.batch * qtiles);
    S = S < long_slices ? S : long_slices;
    Radius rx{};
    rx.slices = static_cast<int>(S);
    rx.radius = radius;
    rx.capacity = cap;
    rx.count = reinterpret_cast<unsigned long long*>(count);
    rx.walked = reinterpret_cast<unsigned long long*>(walked);
    rx.bd = bound_of(prob->p, a.n, a.m);
    // the hits' keys (b P + i) R + j are unique and below 2^end_bit - 1, the key of an unused slot's 0xff..f: a radix
    // sort of the low end_bit bits puts them in torch.nonzero's order, the unused slots last
    int end_bit = 1;
    while (end_bit < 64 && (pairs >> end_bit) != 0) ++end_bit;
    unsigned long long* const keys_out = reinterpret_cast<unsigned long long*>(rows);
    size_t sort_bytes = 0;
    if (cap > 0) {
        const cudaError_t e = cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, rx.keys, keys_out, rx.vals, values,
                                                              cap, 0, end_bit, s);
        if (e != cudaSuccess) return fail(static_cast<int>(e), "radix sort set-up: %s", cudaGetErrorString(e));
    }
    sot::pairwise::Carve c;
    const CdfScratch cs = carve_cdfs(c, a);
    const long long at_eu = c.take(prune ? 8LL * KL * BP : 0), at_du = c.take(prune ? 8LL * BP : 0);
    const long long at_ev = c.take(prune ? 8LL * KL * BR : 0), at_dv = c.take(prune ? 8LL * BR : 0);
    const long long at_keys = c.take(8LL * cap), at_vals = c.take(4LL * cap);
    const long long at_sort = c.take(static_cast<long long>(sort_bytes));
    char* scratch = nullptr;
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&scratch), static_cast<size_t>(c.bytes), s);
    if (e != cudaSuccess) return fail(static_cast<int>(e), "pairwise scratch: %s", cudaGetErrorString(e));
    place_cdfs(a, cs, scratch);
    double* const emb_u = reinterpret_cast<double*>(scratch + at_eu);
    double* const del_u = reinterpret_cast<double*>(scratch + at_du);
    double* const emb_v = reinterpret_cast<double*>(scratch + at_ev);
    double* const del_v = reinterpret_cast<double*>(scratch + at_dv);
    rx.emb_u = emb_u;
    rx.del_u = del_u;
    rx.emb_v = emb_v;
    rx.del_v = del_v;
    rx.keys = reinterpret_cast<unsigned long long*>(scratch + at_keys);
    rx.vals = reinterpret_cast<float*>(scratch + at_vals);
    e = cudaMemsetAsync(rx.keys, 0xff, 8 * static_cast<size_t>(cap), s);  // unused slots sort last
    int rc = e == cudaSuccess ? SOT_OK : fail(static_cast<int>(e), "cudaMemsetAsync: %s", cudaGetErrorString(e));
    if (rc == SOT_OK) rc = launch_cdfs(a, s);
    if (rc == SOT_OK && prune) rc = launch_embed(a, emb_u, del_u, emb_v, del_v, s);
    if (rc == SOT_OK) {
        const long long grid = a.batch * qtiles * S;
        const long long smem = 8LL * (KL * KQ + KQ + KD * KL + KD + 1) +
                               4LL * (pad4(a.n) + pad4(a.m) + 3LL * KQ * KD + 2);
        e = prune ? launch_big<sot_pairwise_radius_kernel<true, false>>(grid, 32 * KW, smem, s, a, rx)
            : cut ? launch_big<sot_pairwise_radius_kernel<false, true>>(grid, 32 * KW, smem, s, a, rx)
                  : launch_big<sot_pairwise_radius_kernel<false, false>>(grid, 32 * KW, smem, s, a, rx);
        rc = sot::launched(e, "sot_pairwise_radius_kernel");
    }
    if (rc == SOT_OK && cap > 0) {
        e = cub::DeviceRadixSort::SortPairs(scratch + at_sort, sort_bytes, rx.keys, keys_out, rx.vals, values, cap, 0,
                                            end_bit, s);
        rc = sot::launched(e, "cub::DeviceRadixSort::SortPairs");
    }
    if (rc == SOT_OK && cap > 0) {
        sot_pairwise_radius_split_kernel<<<static_cast<unsigned>((cap + 255) / 256), 256, 0, s>>>(rx.count, cap,
                                                                                                  a.rows_v, rows, cols);
        rc = sot::launched(cudaGetLastError(), "sot_pairwise_radius_split_kernel");
    }
    return finish(rc, scratch, s);
}

}  // extern "C"
