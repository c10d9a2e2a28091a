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

}  // namespace pairwise
}  // namespace sot

namespace {

using sot::fail;
using sot::pairwise::Args;
using sot::pairwise::pad4;

int validate_pairwise(const sot_pairwise_problem* p) {
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

}  // extern "C"
