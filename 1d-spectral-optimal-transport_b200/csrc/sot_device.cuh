// Device-side building blocks for the SOT kernels (sm_100a).
//
// Nothing here is a port: the reference (`losses.py:129-313`) is a chain of ~30 ATen launches
// (sort / gather / cumsum / cat+sort / searchsorted / take_along_dim / elementwise); these
// helpers implement the same mathematics as ONE pass per frame that never leaves the SM:
// TMA bulk copy -> registers -> packed-fp32 prefix sums with fp64 offsets -> merge-path partition ->
// sequential walk.  (PTX wrappers and the transport cost live here; the kernel is in sot_kernels.cuh.)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define SOT_DEVINL __device__ __forceinline__

namespace sot {

constexpr unsigned FULL_MASK = 0xffffffffu;
constexpr float SAFE_EPS = 1e-7f;          // utils.py:135 (safe_divide eps)
constexpr float FLT_BIG = 3.402823466e+38f;  // FLT_MAX: data clamp so the +inf sentinel stays unique

enum : int {
    FLAG_SQUARE = 1,     // square_dist          losses.py:172-174
    FLAG_CUT_SCALE = 2,  // dont_normalize       losses.py:180-182
    FLAG_LIMIT = 4,      // limit_quantile_range losses.py:306-307
    FLAG_RAW = 8,        // rows are weights used as given (module-level wasserstein_1d, :223-313)
    FLAG_UNIFORM = 16,   // caller asserts: shared supports with pos[i] = pos[0] + i*h EXACTLY in fp32
    FLAG_COMPLEX = 32,   // u, v (and the gradients) are interleaved complex64 STFT rows: |z| is fused in
};

struct FrameArgs {
    const float* u;  // [n_frames, n]  target spectra (or CDF rows)
    const float* v;  // [n_frames, m]  prediction spectra (or CDF rows)
    const float* pos_u;
    const float* pos_v;
    long long pos_u_stride;  // 0: one shared support row; else elements between per-frame rows
    long long pos_v_stride;
    const float* upstream;        // [n_frames] dL_total/dloss_n, or nullptr (= 1)
    const float* upstream_scale;  // device scalar multiplying every upstream value, or nullptr (= 1)
    float upstream_value;         // host constant multiplying every upstream value (1 when unused)
    float* loss;                  // [n_frames] or nullptr
    double* loss_sum;             // device scalar: += sum of the per-frame losses of this launch, or nullptr
    // Mean of the launch finished by its LAST CTA (the reference's closing `torch.mean`, losses.py:211, without
    // a memset, a division or a cast kernel around the launch).  `ticket` (nullable; zero before the launch)
    // counts the CTAs that have added their part to *loss_sum; the last one reads the total, writes
    //   *mean_out = (float)(total * mean_scale)          (nullable)
    //   total_out[0] = total, total_out[1] = post_count  (nullable; what an NCCL all-reduce of the shards sums)
    //   (total, post_count, post_seq) into the mailbox of every peer (post_world > 0; layout of sot_p2p.cu)
    // and leaves *loss_sum = 0, *ticket = 0 for the next launch on the same workspace.
    unsigned int* ticket;
    float* mean_out;
    double mean_scale;
    double* total_out;
    double post_count;
    double* post_mailbox[16];
    int post_world, post_rank;
    unsigned long long post_seq;
    unsigned long long* post_seq_dev;  // nullable: the sequence number lives on the device (*post_seq_dev + 1, stored
                                       // back), so that a CUDA graph holding this launch can be replayed
    float* grad_u;          // [n_frames, n] or nullptr
    float* grad_v;          // [n_frames, m] or nullptr
    // OUT_PLAN outputs, each nullable: [n_frames, n+m] merged grid, un-clamped lower-bound indices
    // and the quantile positions; [n_frames, n] / [n_frames, m] CDF rows
    float* plan_qs;
    int* plan_iu;
    int* plan_iv;
    float* plan_uq;
    float* plan_vq;
    float* plan_cu;
    float* plan_cv;
    long long n_frames;
    int n, m;
    float p;
    int flags;
    // 1.0f and -0.0f as RUN-TIME values (set by the launcher): x * one + neg_zero == x exactly, and because
    // ptxas cannot fold it, a predicated FFMA (fma pipe, two warp-instructions per clock pair) can stand in
    // for an FSEL (alu pipe, half that rate) in the merge walk, which is bound by the alu pipe
    float one, neg_zero, one_b, neg_zero_b;  // (two copies: identical expressions would be merged and re-selected)
};

SOT_DEVINL float f_inf() { return __int_as_float(0x7f800000); }
SOT_DEVINL float f_nan() { return __int_as_float(0x7fc00000); }

// ------------------------------------------------------------------------------------------
// TMA bulk copy (1-D, `cp.async.bulk`, SASS: UBLKCP) + mbarrier plumbing
// ------------------------------------------------------------------------------------------
SOT_DEVINL uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
SOT_DEVINL void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
SOT_DEVINL void fence_mbar_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
SOT_DEVINL void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
SOT_DEVINL void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared, completion counted in bytes on `bar`; all of dst, src, bytes 16-byte aligned
SOT_DEVINL void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// shared -> global
SOT_DEVINL void bulk_s2g(void* dst, const void* src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)),
                 "r"(bytes)
                 : "memory");
}
SOT_DEVINL void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
SOT_DEVINL void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// make generic-proxy shared-memory writes visible to the async (TMA) proxy
SOT_DEVINL void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// |d|^p; PMODE 2 -> d*d compiled in (losses.py:313 with p=2); PMODE 3 -> the same, in a kernel that also has NO cutoff
// mask compiled into its merge walk (limit_quantile_range off: the BASELINE "NoCut" sweep); PMODE 0 -> any p at run time:
// d*d for 2, |d| for 1 (:311-312), powf(|d|, p) otherwise (:313)
template <int PMODE>
SOT_DEVINL float cost_of_gap(float d, float p);

template <int PMODE>
SOT_DEVINL float transport_cost(float pa, float pb, float p) {
    return cost_of_gap<PMODE>(pa - pb, p);
}

template <int PMODE>
SOT_DEVINL float cost_of_gap(float d, float p) {
    // __fmul_rn: never contracted into an FMA with a later subtraction, so |d|^2 is rounded
    // once on its own exactly like the reference's `diff.pow(2)` tensor (losses.py:313)
    if constexpr (PMODE == 2 || PMODE == 3) {
        return __fmul_rn(d, d);
    } else {
        if (p == 2.0f) return __fmul_rn(d, d);
        const float ad = fabsf(d);
        return (p == 1.0f) ? ad : powf(ad, p);
    }
}

// ---- packed fp32x2 arithmetic (sm_100: FADD2 / FMUL2 / FFMA2, two lanes per issued instruction).
// The kernel is bound by instruction issue, so everything that is elementwise on (u, v) bin pairs
// -- squares, local prefix sums, CDF scaling, the gradient chain rule -- runs on pairs.
using f32x2 = unsigned long long;
SOT_DEVINL f32x2 pack2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
SOT_DEVINL void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
SOT_DEVINL f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
SOT_DEVINL f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
SOT_DEVINL f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}

// fp64 reciprocal of a positive float >= 1e-7: hardware approximation + two Newton steps
SOT_DEVINL double recip_f64(float x) {
    const double xd = static_cast<double>(x);
    double r = static_cast<double>(__fdividef(1.0f, x));
    r = fma(r, fma(-xd, r, 1.0), r);
    r = fma(r, fma(-xd, r, 1.0), r);
    return r;
}

// One Hillis-Steele step of a warp scan of an fp64 value that is carried as an EXCLUSIVE scan: the lane at the
// edge (lane 0; lane 31 when REVERSE) holds 0.0 from start to end, so a lane whose partner would lie outside the
// warp reads that lane instead (`src` = clamped partner lane) and adds 0.0 -- an unconditional add.  (A predicated
// fp64 add costs DADD + 2 FSEL + moves after ptxas; `__shfl_up_sync(double)` three times as much.)
SOT_DEVINL void scan_step(double& v, int src) {
    asm volatile(
        "{\n .reg .b32 lo, hi, ylo, yhi;\n .reg .f64 y;\n"
        " mov.b64 {lo, hi}, %0;\n"
        " shfl.sync.idx.b32 ylo, lo, %1, 0x1f, 0xffffffff;\n"
        " shfl.sync.idx.b32 yhi, hi, %1, 0x1f, 0xffffffff;\n"
        " mov.b64 y, {ylo, yhi};\n"
        " add.f64 %0, %0, y;\n}"
        : "+d"(v)
        : "r"(src));
}
// Exclusive scans (prefix; suffix when REVERSE) over the TPF threads of the CTA of two fp32 values, carried
// in fp64.  ta, tb: my values; returns my exclusive offsets and the CTA totals.  One CTA barrier when the
// CTA has more than one warp; `slot` holds 2 * NW doubles.
// nxt_a / nxt_b = the exclusive offset of the NEXT thread (the CTA total for the last one), bitwise: the
// CDF stage caps my entries with it.
template <int TPF, bool REVERSE, bool WANT_NEXT>
SOT_DEVINL void cta_scan2(float ta, float tb, double& off_a, double& off_b, double& nxt_a, double& nxt_b,
                          double& total_a, double& total_b, double* slot, int tid) {
    // TPF < 32 (sub-warp frames: several frames share a warp, each in its own group of TPF lanes): the scan runs
    // inside the group -- `lane` is the position in the group, `base` the warp lane the group starts at.
    constexpr int W = TPF < 32 ? TPF : 32;
    constexpr int NW = (TPF + 31) / 32;
    const int lane = tid & (W - 1), w = tid >> 5;
    const int base = static_cast<int>(threadIdx.x & 31u) - lane;
    const int edge = REVERSE ? W - 1 : 0;  // the lane with nothing before it
    // shift by one lane first: the inclusive scan of the shifted values is the exclusive scan
    float sa = REVERSE ? __shfl_down_sync(FULL_MASK, ta, 1) : __shfl_up_sync(FULL_MASK, ta, 1);
    float sb = REVERSE ? __shfl_down_sync(FULL_MASK, tb, 1) : __shfl_up_sync(FULL_MASK, tb, 1);
    double ea = lane == edge ? 0.0 : static_cast<double>(sa);
    double eb = lane == edge ? 0.0 : static_cast<double>(sb);
#pragma unroll
    for (int off = 1; off < W; off <<= 1) {
        const int src = base + (REVERSE ? min(lane + off, W - 1) : max(lane - off, 0));
        scan_step(ea, src);
        scan_step(eb, src);
    }
    // warp totals, formed on the last lane of the scan direction
    const double wa_mine = ea + static_cast<double>(ta), wb_mine = eb + static_cast<double>(tb);
    if constexpr (NW == 1) {
        off_a = ea;
        off_b = eb;
        total_a = __shfl_sync(FULL_MASK, wa_mine, base + W - 1 - edge);
        total_b = __shfl_sync(FULL_MASK, wb_mine, base + W - 1 - edge);
        if constexpr (WANT_NEXT) {
            const double na = REVERSE ? __shfl_up_sync(FULL_MASK, ea, 1) : __shfl_down_sync(FULL_MASK, ea, 1);
            const double nb = REVERSE ? __shfl_up_sync(FULL_MASK, eb, 1) : __shfl_down_sync(FULL_MASK, eb, 1);
            nxt_a = lane == W - 1 - edge ? total_a : na;
            nxt_b = lane == W - 1 - edge ? total_b : nb;
        }
    } else {
        if (lane == 31 - edge) {
            slot[w] = wa_mine;
            slot[NW + w] = wb_mine;
        }
        __syncthreads();
        double pa = 0.0, pb = 0.0, qa = 0.0, qb = 0.0, xa = 0.0, xb = 0.0;  // prefix before my warp, through my warp, total
#pragma unroll
        for (int k = 0; k < NW; ++k) {
            const int kk = REVERSE ? (NW - 1 - k) : k;
            const double va = slot[kk], vb = slot[NW + kk];
            if (REVERSE ? (kk > w) : (kk < w)) {
                pa = xa + va;
                pb = xb + vb;
            }
            xa += va;
            xb += vb;
            if (kk == w) {
                qa = xa;
                qb = xb;
            }
        }
        off_a = pa + ea;
        off_b = pb + eb;
        total_a = xa;
        total_b = xb;
        if constexpr (WANT_NEXT) {
            // next thread in my warp: its offset is pa + (its ea), the same addition it performs itself; across
            // the warp boundary: the next warp's pa is exactly qa (same sequence of additions), plus its ea = 0
            const double na = REVERSE ? __shfl_up_sync(FULL_MASK, off_a, 1) : __shfl_down_sync(FULL_MASK, off_a, 1);
            const double nb = REVERSE ? __shfl_up_sync(FULL_MASK, off_b, 1) : __shfl_down_sync(FULL_MASK, off_b, 1);
            nxt_a = lane == 31 - edge ? qa : na;
            nxt_b = lane == 31 - edge ? qb : nb;
        }
    }
}

// The same for two fp64 values (raw-weights mode, not a hot path): a, b in = my value, out = exclusive offset.
template <int TPF>
SOT_DEVINL void cta_scan2d(double& a, double& b, double& total_a, double& total_b, double* slot, int tid) {
    constexpr int NW = TPF / 32;
    const int lane = tid & 31, w = tid >> 5;
    double ia = a, ib = b;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const double ya = __shfl_up_sync(FULL_MASK, ia, off), yb = __shfl_up_sync(FULL_MASK, ib, off);
        if (lane >= off) {
            ia += ya;
            ib += yb;
        }
    }
    double ea = __shfl_up_sync(FULL_MASK, ia, 1), eb = __shfl_up_sync(FULL_MASK, ib, 1);
    if (lane == 0) ea = eb = 0.0;
    const double wa = __shfl_sync(FULL_MASK, ia, 31), wb = __shfl_sync(FULL_MASK, ib, 31);
    if constexpr (NW == 1) {
        a = ea;
        b = eb;
        total_a = wa;
        total_b = wb;
    } else {
        if (lane == 0) {
            slot[w] = wa;
            slot[NW + w] = wb;
        }
        __syncthreads();
        double pa = 0.0, xa = 0.0, pb = 0.0, xb = 0.0;
#pragma unroll
        for (int k = 0; k < NW; ++k) {
            const double va = slot[k], vb = slot[NW + k];
            if (k < w) {
                pa = xa + va;
                pb = xb + vb;
            }
            xa += va;
            xb += vb;
        }
        a = pa + ea;
        b = pb + eb;
        total_a = xa;
        total_b = xb;
    }
}

// Called by one thread per CTA after its atomicAdd into *loss_sum: the CTA that draws the last ticket owns the
// total (every other CTA's add is ordered before its ticket by the fence) and finishes the mean -- see FrameArgs.
// Mailbox layout = sot_p2p.cu: slot [rank][phase = seq & 7] of kP2PSlot = 9 doubles, entry [8] = sequence number.
SOT_DEVINL void finish_mean(const FrameArgs& args) {
    __threadfence();
    if (atomicAdd(args.ticket, 1u) != gridDim.x - 1) return;
    __threadfence();
    const double total = __longlong_as_double(static_cast<long long>(
        atomicExch(reinterpret_cast<unsigned long long*>(args.loss_sum), 0ULL)));
    *args.ticket = 0;
    if (args.mean_out != nullptr) *args.mean_out = static_cast<float>(total * args.mean_scale);
    if (args.total_out != nullptr) {
        args.total_out[0] = total;
        args.total_out[1] = args.post_count;
    }
    if (args.post_world > 0) {
        unsigned long long seq = args.post_seq;
        if (args.post_seq_dev != nullptr) {
            seq = *args.post_seq_dev + 1ULL;
            *args.post_seq_dev = seq;
        }
        const int phase = static_cast<int>(seq & 7ULL);
        for (int r = 0; r < args.post_world; ++r) {
            double* dst = args.post_mailbox[r] + (static_cast<long long>(args.post_rank) * 8 + phase) * 9;
            asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(dst), "d"(total) : "memory");
            asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(dst + 1), "d"(args.post_count) : "memory");
        }
        // ONE system-scope fence between the values and the sequence numbers of all peers (a release store per peer
        // is a fence per peer: measured 21 us per step at 8 GPUs against 10 us at 2), then plain stores
        __threadfence_system();
        const double seq_val = static_cast<double>(seq);
        for (int r = 0; r < args.post_world; ++r) {
            double* dst = args.post_mailbox[r] + (static_cast<long long>(args.post_rank) * 8 + phase) * 9;
            asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(dst + 8), "d"(seq_val) : "memory");
        }
    }
}

// Thread 0 of every CTA of a launch that sums its losses: add the CTA's part, the last CTA finishes the mean.
SOT_DEVINL void add_cta_loss(const FrameArgs& args, double cta_loss) {
    atomicAdd(args.loss_sum, cta_loss);
    if (args.ticket != nullptr) finish_mean(args);
}

// ---- per-frame arithmetic of the frame kernel (sot_kernels.cuh) and the split-frame kernel (sot_long.cu): one copy,
// so a row that either kernel can take gets the same bits from both
struct Norm {  // 1/mass of each row, and whether the mass carries gradient
    double inv_u, inv_v;
    bool u_live, v_live;  // mass above the safe_divide floor (utils.py:137: den <= eps -> eps)
};
// tot_u, tot_v: fp64 sums of the accumulated values; cut mode scales v by u's mass; RAW: weights used as given
template <bool RAW>
SOT_DEVINL Norm normalise(double tot_u, double tot_v, bool cut_scale) {
    Norm nm;
    const float mass_u = static_cast<float>(tot_u), mass_v = static_cast<float>(tot_v);
    nm.u_live = mass_u > SAFE_EPS;
    nm.v_live = mass_v > SAFE_EPS;
    nm.inv_u = recip_f64(nm.u_live ? mass_u : SAFE_EPS);
    nm.inv_v = cut_scale ? nm.inv_u : recip_f64(nm.v_live ? mass_v : SAFE_EPS);
    if constexpr (RAW) {
        nm.inv_u = nm.inv_v = 1.0;
        nm.u_live = nm.v_live = false;
    }
    return nm;
}
// false when NaN / inf anywhere (or an overflowing cut-mode scale) poisons the frame
SOT_DEVINL bool finite_frame(double tot_u, double tot_v, const Norm& nm) {
    return (fabs(tot_u * nm.inv_u) <= static_cast<double>(FLT_BIG)) &&
           (fabs(tot_v * nm.inv_v) <= static_cast<double>(FLT_BIG));
}

// Segments of a thread's local prefix sums: 33 sequential fp32 adds leave up to 5 ulp of the fp64 CDF on the paper's
// spectra, four runs of 8 or 9 <= 3, and four short dependency chains issue faster than one long one.
__host__ __device__ constexpr int cdf_segments(int E) { return E >= 25 ? 4 : 1; }
template <int E>
__host__ __device__ constexpr int seg_begin(int s) { return (E * s) / cdf_segments(E); }

// Raw weights: a plain cumsum in fp64 per entry like the reference's (with a handful of atoms the strict `qs > 1` mask
// decides over a whole atom on the last ulp).  ru, rv: my exclusive offsets in, plus my sums out.
template <int E, typename StoreU, typename StoreV>
SOT_DEVINL void raw_cumsum(const f32x2 (&x2)[E], bool sq, double& ru, double& rv, const StoreU& store_u,
                           const StoreV& store_v) {
#pragma unroll
    for (int c = 0; c < E; ++c) {
        float a, b;
        unpack2(x2[c], a, b);
        ru += static_cast<double>(sq ? a * a : a);
        rv += static_cast<double>(sq ? b * b : b);
        store_u(c, static_cast<float>(ru));
        store_v(c, static_cast<float>(rv));
    }
}

// CDF entry = fminf(head + fma(local prefix, 1/mass, ride), cap).  (head, tail): fp32 split of (sum of the threads
// before me) * 1/mass, so that the one rounding that matters is the final add; cap: the next thread's head, bitwise,
// which keeps the row non-decreasing across threads.  Segments restart the prefix and ride on the pre-head value of
// the previous segment's last entry (the tail in the first): monotone in the prefix, so also across segments.
struct CdfScale {
    f32x2 head, tail, inv;
    float cap_u, cap_v;
};
SOT_DEVINL CdfScale cdf_scale(double off_u, double off_v, double nxt_u, double nxt_v, const Norm& nm) {
    const double base_u = off_u * nm.inv_u, base_v = off_v * nm.inv_v;
    const float bh_u = static_cast<float>(base_u), bh_v = static_cast<float>(base_v);
    const float bl_u = static_cast<float>(base_u - static_cast<double>(bh_u));
    const float bl_v = static_cast<float>(base_v - static_cast<double>(bh_v));
    return {pack2(bh_u, bh_v), pack2(bl_u, bl_v), pack2(static_cast<float>(nm.inv_u), static_cast<float>(nm.inv_v)),
            static_cast<float>(nxt_u * nm.inv_u), static_cast<float>(nxt_v * nm.inv_v)};
}
// SQ: x^2 fused into the add.  store_u(c, entry), store_v(c, entry): one per side, in this order (the frame kernel's
// stores are volatile asm).
template <bool SQ, int E, typename StoreU, typename StoreV>
SOT_DEVINL void cdf_entries(const f32x2 (&x2)[E], const CdfScale& k, const StoreU& store_u, const StoreV& store_v) {
    f32x2 ride = k.tail;
#pragma unroll
    for (int s = 0; s < cdf_segments(E); ++s) {
        f32x2 p2 = 0, in2 = ride;
#pragma unroll
        for (int c = seg_begin<E>(s); c < seg_begin<E>(s + 1); ++c) {
            p2 = SQ ? fma2(x2[c], x2[c], p2) : add2(p2, x2[c]);
            in2 = fma2(p2, k.inv, ride);
            float ca, cb;
            unpack2(add2(in2, k.head), ca, cb);
            store_u(c, fminf(ca, k.cap_u));
            store_v(c, fminf(cb, k.cap_v));
        }
        ride = in2;
    }
}

// Tie-group rule of the gradient walk at a slot of value q: dL/dCDF of `consumed` (the entry the slot before took) is
// (m*d)_group - (m*d)_next group at a group's last slot, else 0.  md_new: m*d of a group starting here, masked.  A
// group opened before my chunk (`inherited`, m*d unknown) that closes here leaves `consumed` in `fix` for look_back.
template <typename Idx>
SOT_DEVINL float tie_step(float q, float qprev, float md_new, Idx consumed, float& md_prev, bool& inherited, Idx& fix) {
    const bool same = (q == qprev);
    const float md = same ? md_prev : md_new;
    const float g = md_prev - md;
    fix = (inherited && !same) ? consumed : fix;
    inherited = inherited && same;
    md_prev = md;
    return g;
}

// From `at` back by `step`: the first per-chunk carry that is not the marker (< 0: "my whole chunk continues a group
// opened before it"; chunk 0 never carries it)
template <typename Idx, typename Load>
SOT_DEVINL auto look_back(Idx at, Idx step, Load load) {
    auto c = load(at);
    while (c < 0) {
        at -= step;
        c = load(at);
    }
    return c;
}

// Chain rule of the normalisation: dot = sum_i gw_i w_i / mass; a clamped mass has no derivative (torch.where)
SOT_DEVINL void mass_terms(const Norm& nm, bool cut_scale, double dot_u, double dot_v, double& corr_u, double& corr_v) {
    corr_u = nm.u_live ? (cut_scale ? dot_u + dot_v : dot_u) : 0.0;
    corr_v = (!cut_scale && nm.v_live) ? dot_v : 0.0;
}
// dL_total / dloss of a frame
SOT_DEVINL float upstream_of(const FrameArgs& args, long long frame) {
    return (args.upstream != nullptr ? args.upstream[frame] : 1.0f) *
           (args.upstream_scale != nullptr ? *args.upstream_scale : 1.0f) * args.upstream_value;
}
// Factors of the gradient rows: 1/mass x upstream (x 2 for square_dist), NaN for a poisoned frame
SOT_DEVINL void grad_scale(const Norm& nm, float up, bool square, bool finite, float& ku, float& kv) {
    ku = finite ? static_cast<float>(nm.inv_u) * up * (square ? 2.0f : 1.0f) : f_nan();
    kv = finite ? static_cast<float>(nm.inv_v) * up * (square ? 2.0f : 1.0f) : f_nan();
}

}  // namespace sot
