// SOT frame kernel: per-frame 1-D Wasserstein (W_p^p) between two spectra, forward and
// fused forward+backward.  ONE FRAME PER CTA of TPF threads, persistent grid, many CTAs per SM.
//
// Reference semantics reproduced (file:line into /root/reference):
//   losses.py:172-184  square, mass, safe_divide (cut mode divides the prediction by the
//                      TARGET's mass), utils.py:135-142
//   losses.py:292-293  inclusive CDFs                     -> packed-fp32 local prefix sums, fp64 scan of the
//                                                           per-thread sums (raw weights: fp64 per entry)
//   losses.py:295      sort(cat(cu, cv))                  -> merge-path partition + sequential walk
//   losses.py:214-220  searchsorted-left + clamp + gather -> running co-ranks of the walk
//   losses.py:301-313  sum_k dq_k * |uq_k - vq_k|^p, strict `qs > 1` mask
//   autograd of all of the above (SURVEY.md 3.3)          -> dL/dCDF array, suffix scans,
//                                                           normalisation chain rule, 2x
//
// Shared memory: first the small per-CTA structures (scan scratch, one carry per chunk, mbarrier), then rows of
// RS >= TPF * E + 8 floats at COMPILE-TIME offsets, so that for a CDF entry at shared
// address a its support position is at a + POS_OFF and its dL/dCDF at a + G_OFF (immediates):
//   rows 0, 1 : CDF of u / v, entry [n] / [m] = +inf sentinel
//   rows 2, 3 : support positions of u / v, entry [n] / [m] repeats the last one (the reference's
//               clamp of the searchsorted index, losses.py:220); written once per CTA when the
//               support is shared by all frames.  (A single row for u and v when they share the
//               grid was tried: more resident CTAs, no speed-up -- the kernel is bound by shared-
//               memory wavefronts, not by occupancy.)
//               UNIFORM GRIDS (template flag UNI; every linear-frequency config): positions are
//               pos[0] + i*h exactly, so these two rows and the position load of every merged slot
//               disappear -- the position difference of the two heads is tracked with exact +-h steps.
//   next 2    : (gradient kernel) dL/dCDF of u / v
//   next 4    : (complex input, template flag CPLX) the two interleaved complex64 STFT rows: the
//               magnitude (squared) is formed while they are read -- no |.| tensor in HBM -- and the
//               gradient kernel overwrites them in place with the complex gradient rows
//   then      : 64 bytes of padding.  Every thread loads and stores all E entries of its bins without guards: the
//               rows are long enough, what lies past the end of the data is masked once (stage 1) or overwritten
//               by the threads that own it (sentinels, zeroed dL/dCDF tail)
// The raw rows of a frame arrive by TMA bulk copy (`cp.async.bulk`, SASS UBLKCP).  A 4*n-byte row
// is only 4-byte aligned (n = 1025 / 257), the bulk unit is 16 bytes: the copy therefore fetches
// the 16-byte aligned WINDOW around the row and the kernel skips the `lead` bytes in front.  The
// landing zone is rows 0/1: each thread has its bins in registers before the CDF is written in
// place, and the next frame is prefetched as soon as the last reader of the CDF rows is done.
// Gradient rows leave the same way: written over the dL/dCDF rows at the row's own 16-byte phase,
// bulk store of the aligned middle, <= 3 scalar stores per edge.
// Thread t owns the E consecutive bins [t*E, t*E+E) of both rows ("blocked"); E is odd so every
// blocked access of a warp is bank-conflict free.  Everything elementwise runs on (u, v) PAIRS in
// packed fp32x2 instructions (FFMA2 / FADD2 / FMUL2); the merge walk keeps its selects and masks on
// the fma pipe (predicated FFMA, FFMA.SAT) because the alu pipe runs at half rate.
#pragma once
#include <type_traits>

#include "sot_device.cuh"

namespace sot {

enum : int {
    MODE_SPECTRA = 0,  // inputs are magnitudes: full prologue
    MODE_RAW = 2,      // inputs are weights used as given (FLAG_RAW): no normalisation, CDF = cumsum with fp64
                       // accumulation exactly like the reference's (see stage 2)
    MODE_CDF = 1,      // inputs are CDF rows (parity harness): skip the prologue; with grads the
                       // outputs are dL/dcu, dL/dcv (no suffix scan / chain rule)
};

enum : int {
    OUT_LOSS = 0,  // per-frame loss only (forward)
    OUT_GRAD = 1,  // loss + gradient rows (fused forward+backward)
    OUT_PLAN = 2,  // loss + the transport plan: qs, searchsorted indices, quantiles, CDFs
                   // (`return_quantiles=True`, losses.py:198-201, 299-300; also the parity harness)
};

// ---- compile-time shared-memory layout ---------------------------------------------------------
template <int TPF, int RS, int OUT, int NCH, bool UNI, bool CPLX>
struct Layout {
    static constexpr uint32_t ROW = 4u * RS;
    // small per-CTA structures first, the rows after them: a thread whose bins lie past the end of a row reads
    // (and masks) whatever follows -- after the last row that is the PAD below, never live scratch data
    static constexpr uint32_t SCRATCH = 0;                        // 8 doubles per warp
    static constexpr uint32_t CARRY = SCRATCH + 64u * ((TPF + 31) / 32);  // m*d of the group open at the end of each chunk
    static constexpr uint32_t MBAR = (CARRY + 4u * NCH * TPF + 15u) & ~15u;
    static constexpr uint32_t HEAD = (MBAR + 16u + 127u) & ~127u;
    static constexpr uint32_t A = HEAD, B = HEAD + ROW;  // CDF rows (also the landing zone of the raw rows)
    static constexpr uint32_t POS_OFF = 2 * ROW;  // cdf address -> position address (two rows; none when UNI)
    static constexpr uint32_t PROWS = UNI ? 0 : 2;
    static constexpr uint32_t G_OFF = (2 + PROWS) * ROW;  // cdf address -> dL/dCDF address (two rows; also output staging)
    // (A separate landing zone for the raw rows, so that the next frame is fetched a whole frame ahead, was
    // measured twice -- on the shared-memory-bound v3 kernel and again on the packed-fp32 one: the mbarrier
    // wait disappears from the stall samples, the run time does not change (other resident CTAs fill the
    // wait) -- so the rows stay in place and the shared memory goes to resident CTAs.)
    // Complex (STFT) input: the raw rows are twice as wide, land in their own two double rows and, in the
    // gradient kernel, are overwritten in place by the complex gradient rows (= output staging).
    static constexpr uint32_t REAL_ROWS = 2 + PROWS + ((OUT == OUT_GRAD) ? 2 : 0);
    static constexpr uint32_t LAND = CPLX ? HEAD + REAL_ROWS * ROW : A;
    static constexpr uint32_t LAND_ROW = CPLX ? 2 * ROW : ROW;  // bytes between the u and the v landing row
    static constexpr uint32_t ROWS = REAL_ROWS + (CPLX ? 4 : 0);
    static constexpr uint32_t PAD = 64u;  // (rows hold TPF * E entries and the lead: nothing is read past the last row)
    static constexpr uint32_t TOTAL = HEAD + ROWS * ROW + PAD;
    // sub-warp frames: one such block per frame of the CTA, 16 banks apart -- the 16 lanes of a frame touch 16 of the
    // 32 banks in every blocked access (17 t mod 32), the other frame of the warp gets the other 16
    static constexpr uint32_t SLOT = ((TOTAL + 127u) & ~127u) + 64u;
    static constexpr int MAX_BINS = RS - 7;  // sentinel + up to 3 floats of lead + rounding of the bulk window
};

// ---- raw shared-memory access by 32-bit shared address (exact instructions, no generic ptrs) ---
SOT_DEVINL float lds32(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
template <uint32_t OFF>
SOT_DEVINL float lds32o(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1+%2];" : "=f"(v) : "r"(a), "n"(OFF));
    return v;
}
SOT_DEVINL void sts32(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
template <uint32_t OFF>
SOT_DEVINL void sts32o(uint32_t a, float v) {
    asm volatile("st.shared.f32 [%0+%2], %1;" ::"r"(a), "f"(v), "n"(OFF) : "memory");
}
SOT_DEVINL void lds64(uint32_t a, float& x, float& y) {
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(x), "=f"(y) : "r"(a));
}
SOT_DEVINL void sts64(uint32_t a, float x, float y) {
    asm volatile("st.shared.v2.f32 [%0], {%1, %2};" ::"r"(a), "f"(x), "f"(y) : "memory");
}
// (lo, hi) = (shared[a], shared[b]): the loads define the two halves of the pair directly
SOT_DEVINL f32x2 lds32x2(uint32_t a, uint32_t b) {
    f32x2 r;
    asm volatile("{\n .reg .f32 lo, hi;\n ld.shared.f32 lo, [%1];\n ld.shared.f32 hi, [%2];\n mov.b64 %0, {lo, hi};\n}"
                 : "=l"(r)
                 : "r"(a), "r"(b));
    return r;
}
// (keep_lo ? lo : 0, keep_hi ? hi : 0)
SOT_DEVINL f32x2 mask2(f32x2 v, bool keep_lo, bool keep_hi) {
    f32x2 r;
    asm("{\n .reg .f32 lo, hi;\n .reg .pred p, q;\n mov.b64 {lo, hi}, %1;\n setp.ne.s32 p, %2, 0;\n setp.ne.s32 q, %3, 0;\n"
        " selp.f32 lo, lo, 0f00000000, p;\n selp.f32 hi, hi, 0f00000000, q;\n mov.b64 %0, {lo, hi};\n}"
        : "=l"(r)
        : "l"(v), "r"(static_cast<int>(keep_lo)), "r"(static_cast<int>(keep_hi)));
    return r;
}
// One merge step's advance: the consumed side (v if b < a, else u: u first on equal values, the
// stable order of `cat(cu, cv)`) gets its next CDF entry and that entry's position.  ONE load per
// array from the SELECTED address: a pair of predicated loads (one per side, half the lanes each)
// costs a shared-memory wavefront per instruction, and wavefronts are what bounds this kernel.
// `consumed` = address of the CDF entry that was taken.  POS4 = POS_OFF + 4.
// The value selects are predicated FFMAs (x * one + neg_zero with run-time 1.0f / -0.0f, see FrameArgs): the
// walk is bound by the alu pipe (FSEL / FSETP / FMNMX / integer adds, one warp-instruction per two clocks)
// while the fma pipe has room; `k` = the four constants.
struct WalkConsts {
    float one, nz, one_b, nz_b;
};
template <uint32_t POS4>
SOT_DEVINL void advance(float& a, float& pa, float& b, float& pb, uint32_t& adrA, uint32_t& adrB,
                        uint32_t& consumed, const WalkConsts& k) {
    asm volatile(
        "{\n"
        ".reg .pred tv;\n"
        ".reg .f32 nv, np;\n"
        "setp.lt.f32 tv, %2, %0;\n"
        "selp.u32 %6, %5, %4, tv;\n"
        "ld.shared.f32 nv, [%6+4];\n"
        "ld.shared.f32 np, [%6+%7];\n"
        "@tv  add.u32 %5, %5, 4;\n"
        "@!tv add.u32 %4, %4, 4;\n"
        "@tv  fma.rn.f32 %2, nv, %8, %9;\n"
        "@tv  fma.rn.f32 %3, np, %8, %9;\n"
        "@!tv fma.rn.f32 %0, nv, %10, %11;\n"
        "@!tv fma.rn.f32 %1, np, %10, %11;\n"
        "}"
        : "+f"(a), "+f"(pa), "+f"(b), "+f"(pb), "+r"(adrA), "+r"(adrB), "=&r"(consumed)
        : "n"(POS4), "f"(k.one), "f"(k.nz), "f"(k.one_b), "f"(k.nz_b));
}
// Uniform-grid advance: no position load; `d` = pos_u[head] - pos_v[head] moves by exactly +h when u
// advances and -h when v advances -- except onto the +inf sentinel, whose position repeats the last
// one (the reference's index clamp).
SOT_DEVINL void advance_uni(float& a, float& d, float& b, uint32_t& adrA, uint32_t& adrB, uint32_t& consumed,
                            float h, float neg_h, const WalkConsts& k) {
    asm volatile(
        "{\n"
        ".reg .pred tv;\n"
        ".reg .f32 nv, dh, live;\n"
        "setp.lt.f32 tv, %2, %0;\n"
        "selp.u32 %5, %4, %3, tv;\n"
        "ld.shared.f32 nv, [%5+4];\n"
        "@tv  add.u32 %4, %4, 4;\n"
        "@!tv add.u32 %3, %3, 4;\n"
        "selp.f32 dh, %7, %6, tv;\n"
        "sub.rn.sat.f32 live, 0f7F7FFFFF, nv;\n"  // 1 for a CDF entry, 0 for the +inf sentinel
        "@tv  fma.rn.f32 %2, nv, %8, %9;\n"
        "@!tv fma.rn.f32 %0, nv, %10, %11;\n"
        "fma.rn.f32 %1, dh, live, %1;\n"
        "}"
        : "+f"(a), "+f"(d), "+f"(b), "+r"(adrA), "+r"(adrB), "=&r"(consumed)
        : "f"(h), "f"(neg_h), "f"(k.one), "f"(k.nz), "f"(k.one_b), "f"(k.nz_b));
}

// One step of the merge-path bit descent, branch free: probe co-rank min(cur + STEP, hi) -- clamping instead of
// skipping keeps the descent correct (the predicate "A[i-1] <= B[k0-i]" is monotone in i: once hi itself passes,
// every later probe is hi again) and every probe address valid, so the two loads need no guard (a guarded pair
// costs BSSY / BSYNC / BRA per step and branch-resolving stalls over 11 dependent rounds).
// sum = addr(A[i]) + addr(B[k0-i]), constant along a diagonal.
template <int STEP>
SOT_DEVINL void search_step(uint32_t& cur, uint32_t hi, uint32_t sum) {
    const uint32_t cand = min(cur + 4u * STEP, hi);
    const float av = lds32(cand - 4);    // A[i-1] for the candidate i (i = lo = 0 is never probed: cand > cur >= A0
    const float bv = lds32(sum - cand);  //  unless hi == cur, and then the row's left neighbour in shared memory is read
    cur = (av <= bv) ? cand : cur;       //  and the outcome is the same position)
}
// the whole descent for NCH interleaved searches: steps TOP, TOP/2, ..., 1 (elements)
template <int STEP, int NCH>
SOT_DEVINL void search_descent(uint32_t (&cur)[NCH], const uint32_t (&hi)[NCH], const uint32_t (&sum)[NCH]) {
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) search_step<STEP>(cur[ch], hi[ch], sum[ch]);
    if constexpr (STEP > 1) search_descent<STEP / 2, NCH>(cur, hi, sum);
}

template <int TPF>
SOT_DEVINL void cta_sync() {
    if constexpr (TPF <= 32) {  // one warp per CTA (TPF < 32: sub-warp frames, several frames in the warp)
        __syncwarp();
    } else {
        __syncthreads();
    }
}

// Resident CTAs per SM requested from ptxas: as many as the shared-memory footprint allows,
// within a sane register budget (forward >= 40, gradient >= 64 registers per thread).
constexpr int min_ctas(int tpf, int e, int smem_bytes, int out) {
    const int by_smem = (227 * 1024) / (smem_bytes + 1024);
#ifndef SOT_REGS_GRAD_E17  // (tuning experiments: -DSOT_REGS_GRAD_E17=.. -DSOT_REGS_LOSS_E17=..)
#define SOT_REGS_GRAD_E17 96
#endif
#ifndef SOT_REGS_LOSS_E17
#define SOT_REGS_LOSS_E17 64
#endif
#ifndef SOT_REGS_GRAD_SUB
#define SOT_REGS_GRAD_SUB 128  // one-warp CTAs with 17 bins per thread (sub-warp frames): no spills
#endif
#ifndef SOT_REGS_GRAD_E9
#define SOT_REGS_GRAD_E9 128  // one warp per frame (n_fft 512): 64 -> 128 registers = no spills, +11 % (profiles/r02_tuning.txt)
#endif
    const int regs = out == OUT_GRAD ? (e <= 9 ? (tpf == 32 ? SOT_REGS_GRAD_E9 : 64)
                                              : (e <= 17 ? (tpf == 32 ? SOT_REGS_GRAD_SUB : SOT_REGS_GRAD_E17) : 168))
                                     : (e <= 9 ? 40 : (e <= 17 ? (tpf == 32 ? 96 : SOT_REGS_LOSS_E17) : 128));
    const int by_regs = 65536 / (tpf * regs);
    const int c = by_smem < by_regs ? by_smem : by_regs;
    return c < 1 ? 1 : (c > 32 ? 32 : c);
}
__host__ __device__ constexpr int ilog2_ceil(int x) {
    int b = 0;
    while ((1 << b) < x) ++b;
    return b;
}

// 16-byte aligned window around row `f` of a [frames, width] fp32 array: `lead` bytes (0, 4, 8, 12)
// sit between the window start and the row.  Only the low address bits matter for the phase, so
// every thread gets it with a few 32-bit operations; the elected thread builds the 64-bit source.
SOT_DEVINL uint32_t row_lead(const float* base, long long f, int width) {
    return (static_cast<uint32_t>(reinterpret_cast<uintptr_t>(base)) +
            4u * static_cast<uint32_t>(width) * static_cast<uint32_t>(f)) & 15u;
}
// the window of row f lies inside the array (safe to fetch with a bulk copy): always true except
// for the first row of an array that does not start, and the last row of one that does not end,
// on a 16-byte boundary
SOT_DEVINL bool row_is_bulk(const float* base, long long f, int width, long long frames) {
    const uint32_t lo = static_cast<uint32_t>(reinterpret_cast<uintptr_t>(base));
    const bool head_ok = (f > 0) || ((lo & 15u) == 0);
    const bool tail_ok = (f + 1 < frames) ||
                         (((lo + 4u * static_cast<uint32_t>(width) * static_cast<uint32_t>(frames)) & 15u) == 0);
    return head_ok && tail_ok;
}

template <int N>
using IC = std::integral_constant<int, N>;

// FPW > 1 ("sub-warp frames", short rows): TPF < 32 threads per frame and FPW = 32 / TPF frames per CTA, each frame in
// its own group of TPF lanes of the one warp with its own block of shared memory, mbarrier and bulk copies.  Every
// lane runs the same instruction stream on its own frame, so the per-frame fixed costs (scans, merge-path search,
// reductions, bookkeeping) are paid once per warp for FPW frames.  Spectra -> loss / gradients only.
template <int TPF, int E, int RS, int NCH, bool UNI, bool CPLX, int PMODE, int OUT, int MODE, int FPW = 1>
__global__ void __launch_bounds__(TPF * FPW, min_ctas(TPF * FPW, E, FPW * Layout<TPF, RS, OUT, NCH, UNI, CPLX>::SLOT, OUT))
    sot_frame_kernel(const FrameArgs args) {
    static_assert(NCH == 1 || NCH == 2, "one or two merge chains per thread");
    constexpr bool SUB = FPW > 1;
    // PMODE 3: p = 2 and no quantile cutoff -- the walk's per-slot mask (FFMA.SAT + FMUL, 2 of its 24 instructions per
    // merged slot) is not compiled in; results are bit-identical to PMODE 2 run without FLAG_LIMIT (keep == 1 there)
    constexpr bool NOLIM = (PMODE == 3);
    static_assert(!NOLIM || (UNI && !CPLX && MODE == MODE_SPECTRA && OUT != OUT_PLAN),
                  "no-cutoff walk: uniform grid, real spectra, loss / gradient outputs");
    static_assert(!SUB || (TPF * FPW == 32 && !CPLX && MODE == MODE_SPECTRA && OUT != OUT_PLAN),
                  "sub-warp frames: one warp per CTA, real spectra, loss / gradient outputs");
    static_assert(RS >= TPF * E + 8, "rows hold every thread's E entries (stored without guards) plus the lead / sentinel");
    static_assert(!(UNI && OUT == OUT_PLAN), "the plan emitter always reads positions");
    static_assert(!CPLX || (MODE == MODE_SPECTRA && OUT != OUT_PLAN), "complex input: loss / gradient from spectra only");
    constexpr bool FROM_BINS = (MODE != MODE_CDF);  // spectra or raw weights: the kernel builds the CDFs
    using LY = Layout<TPF, RS, OUT, NCH, UNI, CPLX>;
    constexpr int CW = CPLX ? 2 : 1;  // floats per raw bin
    constexpr int NCHUNK = NCH * TPF;
    constexpr bool WITH_GRAD = (OUT == OUT_GRAD);
    constexpr int NW = (TPF + 31) / 32;
    constexpr int WG = TPF < 32 ? TPF : 32;  // lanes of a warp that work on one frame
    constexpr int SEARCH_TOP = 1 << (ilog2_ceil(TPF * E + 1) - 1);
    constexpr uint32_t NO_FIX = 0xffffffffu;
    constexpr uint32_t POS4 = LY::POS_OFF + 4;
    constexpr uint32_t LAND = LY::LAND;  // landing zone rows (u, then v at + ROW)
    extern __shared__ __align__(128) unsigned char smem_cta[];
    const int fslot = SUB ? static_cast<int>(threadIdx.x) / TPF : 0;  // which frame of the CTA I work on
    unsigned char* const smem = smem_cta + fslot * LY::SLOT;

    const int n = args.n, m = args.m, K = n + m;
    const bool square = args.flags & FLAG_SQUARE;
    const bool cut_scale = args.flags & FLAG_CUT_SCALE;
    const bool pos_shared = (args.pos_u_stride == 0) && (args.pos_v_stride == 0);
    // contributions with q above `thr` are dropped: the strict `qs > 1` mask (losses.py:307) when
    // limiting, otherwise nothing a real slot can reach
    const float thr = (args.flags & FLAG_LIMIT) ? 1.0f : FLT_BIG;
    // the same test on the fma pipe: keep(q) = sat((thr+ - q) * 2^60) is exactly 1 for q <= thr and 0 above
    // (thr+ = the float after thr; without a limit the constant is +inf and keep == 1 for every finite q)
    const float keep_c = (args.flags & FLAG_LIMIT) ? 1.00000011920928955078125f * 1152921504606846976.0f
                                                   : __int_as_float(0x7f800000);
    const WalkConsts wk{args.one, args.neg_zero, args.one_b, args.neg_zero_b};
    const uint32_t sb = smem_u32(smem);
    const uint32_t A0 = sb + LY::A, B0 = sb + LY::B;

    const int tid = SUB ? static_cast<int>(threadIdx.x) % TPF : static_cast<int>(threadIdx.x);  // within my frame
    const int e0 = tid * E;
    float* const fsm = reinterpret_cast<float*>(smem);
    double* const scratch = reinterpret_cast<double*>(smem + LY::SCRATCH);
    // ONE mbarrier per CTA -- also with several frames per warp: lanes that spin on different barriers leave the
    // (hand-written) wait loop at different times and the warp stays diverged, every later shuffle takes the slow path
    uint64_t* const mbar = reinterpret_cast<uint64_t*>(smem_cta + LY::MBAR);
    const bool elected = SUB ? (threadIdx.x == 0) : (tid == 0);  // issues the bulk loads of the CTA
    const uint32_t carry = sb + LY::CARRY;
    const bool in_u = e0 + E <= n, in_v = e0 + E <= m;  // all of my E bins exist (no guards needed)

    // The K merged slots are cut into NCH * TPF chunks of L consecutive slots; thread t walks chunks
    // NCH*t .. NCH*t + NCH-1 AT THE SAME TIME (NCH independent dependency chains: the walk is a chain of
    // dependent shared-memory loads, and with few resident warps instruction-level parallelism is what
    // hides their latency).  L is ODD on purpose: for a balanced merge chunk c starts near entry L*c/2
    // of each row, and an even L would put the lanes of a warp on few distinct banks (measured: 8-way
    // conflicts on every load of the walk); odd L spreads them.
    const int L = ((K + NCHUNK - 1) / NCHUNK) | 1;
    int k0[NCH], cnt[NCH];
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
        k0[ch] = min((NCH * tid + ch) * L, K);
        cnt[ch] = min(L, K - k0[ch]);  // non-increasing in the chunk index
    }

    if (elected) {
        mbar_init(mbar, 1);
        fence_mbar_init();
    }
    float pu0 = 0.0f, pv0 = 0.0f, hstep = 0.0f;  // (UNI) pos_u[i] = pu0 + i*hstep, pos_v[j] = pv0 + j*hstep
    if constexpr (UNI) {
        pu0 = args.pos_u[0];
        pv0 = args.pos_v[0];
        hstep = args.pos_u[1] - pu0;
    } else if (pos_shared) {  // positions once per CTA
        for (int idx = tid; idx <= n; idx += TPF) fsm[(LY::A + LY::POS_OFF) / 4 + idx] = args.pos_u[min(idx, n - 1)];
        for (int idx = tid; idx <= m; idx += TPF) fsm[(LY::B + LY::POS_OFF) / 4 + idx] = args.pos_v[min(idx, m - 1)];
    }
    (void)pu0;
    (void)pv0;
    (void)hstep;
    __syncthreads();

    const int wu = CW * n, wv = CW * m;  // floats per raw row
    // bulk loads of the frames of one CTA iteration (base frame b): raw rows -> landing rows, one expect_tx
    auto issue_load = [&](long long b) {  // the elected thread
        uint32_t total = 0;
#pragma unroll
        for (int g = 0; g < FPW; ++g) {
            const long long f = SUB ? min(b + g, args.n_frames - 1) : b;
            total += ((row_lead(args.u, f, wu) + 4u * wu + 15u) & ~15u) + ((row_lead(args.v, f, wv) + 4u * wv + 15u) & ~15u);
        }
        mbar_expect_tx(mbar, total);
#pragma unroll
        for (int g = 0; g < FPW; ++g) {
            const long long f = SUB ? min(b + g, args.n_frames - 1) : b;
            const uint32_t lu = row_lead(args.u, f, wu), lv = row_lead(args.v, f, wv);
            const uint32_t bu = (lu + 4u * wu + 15u) & ~15u, bv = (lv + 4u * wv + 15u) & ~15u;
            unsigned char* const dst = smem_cta + g * LY::SLOT + LAND;
            bulk_g2s(dst, reinterpret_cast<const char*>(args.u + f * wu) - lu, bu, mbar);
            bulk_g2s(dst + LY::LAND_ROW, reinterpret_cast<const char*>(args.v + f * wv) - lv, bv, mbar);
        }
    };
    // do ALL frames of the CTA iteration with base frame b come by bulk copy?  (warp uniform)
    auto all_bulk = [&](long long b) {
        bool ok = true;
#pragma unroll
        for (int g = 0; g < FPW; ++g) {
            const long long f = SUB ? min(b + g, args.n_frames - 1) : b;
            ok = ok && row_is_bulk(args.u, f, wu, args.n_frames) && row_is_bulk(args.v, f, wv, args.n_frames);
        }
        return ok;
    };

    // Frames of this CTA: blockIdx.x * FPW + fslot, then + gridDim.x * FPW.  The loop condition is the one of frame
    // slot 0 (warp uniform); a slot that has run out of frames redoes the LAST frame of the batch in lock step
    // (identical values to identical addresses) and keeps it out of the sums (`active`).
    const long long fstride = static_cast<long long>(gridDim.x) * FPW;
    long long fbase = static_cast<long long>(blockIdx.x) * FPW;
    auto frame_of = [&](long long b) { return SUB ? min(b + fslot, args.n_frames - 1) : b; };
    long long frame = frame_of(fbase);
    uint32_t parity = 0;
    double cta_loss = 0.0;  // (thread 0) sum of the losses of the frames this CTA processed
    // state of the frame in flight: phases of its two rows and whether it comes by bulk copy
    uint32_t lead_in_u = 0, lead_in_v = 0;
    bool bulk_in = false;
    if (fbase < args.n_frames) {
        lead_in_u = row_lead(args.u, frame, wu);
        lead_in_v = row_lead(args.v, frame, wv);
        bulk_in = all_bulk(fbase);
        if (bulk_in && elected) issue_load(fbase);
    }

    for (; fbase < args.n_frames; fbase += fstride) {
        frame = frame_of(fbase);
        const bool active = !SUB || (fbase + fslot < args.n_frames);
        // ---- stage 0: the frame's raw rows are (or get) in the landing zone ----------------------
        uint32_t rawU = sb + LAND + 4u * CW * e0, rawV = sb + LAND + LY::LAND_ROW + 4u * CW * e0;  // my first raw bins
        uint32_t cur_lead_u = 0, cur_lead_v = 0;  // phase of this frame's raw rows inside the landing rows
        if (bulk_in) {
            mbar_wait(mbar, parity);
            parity ^= 1;
            cur_lead_u = lead_in_u;
            cur_lead_v = lead_in_v;
            rawU += lead_in_u;
            rawV += lead_in_v;
        } else {  // first / last row of an array whose ends are not 16-byte aligned: plain coalesced loads
            const float* gu = args.u + frame * wu;
            const float* gv = args.v + frame * wv;
            if constexpr (CPLX && OUT == OUT_GRAD) cta_sync<TPF>();  // thread 0 has seen the previous store drain
            for (int idx = tid; idx < wu; idx += TPF) fsm[LAND / 4 + idx] = gu[idx];
            for (int idx = tid; idx < wv; idx += TPF) fsm[(LAND + LY::LAND_ROW) / 4 + idx] = gv[idx];
            cta_sync<TPF>();
        }
        (void)cur_lead_u;
        (void)cur_lead_v;
        // the frame after this one (its load is issued further down, when the landing zone is free)
        const long long next = frame_of(fbase + fstride);
        const bool has_next = fbase + fstride < args.n_frames;  // (warp uniform)
        if (has_next) {
            lead_in_u = row_lead(args.u, next, wu);
            lead_in_v = row_lead(args.v, next, wv);
            bulk_in = all_bulk(fbase + fstride);
        }
        if (!UNI && !pos_shared) {  // per-frame supports
            const float* gpu = args.pos_u + frame * args.pos_u_stride;
            const float* gpv = args.pos_v + frame * args.pos_v_stride;
            for (int idx = tid; idx <= n; idx += TPF) fsm[(LY::A + LY::POS_OFF) / 4 + idx] = gpu[min(idx, n - 1)];
            for (int idx = tid; idx <= m; idx += TPF) fsm[(LY::B + LY::POS_OFF) / 4 + idx] = gpv[min(idx, m - 1)];
        }

        float acc[NCH] = {};  // my part of the frame's loss
        bool finite = true;  // masses (and the scaled totals) are finite numbers
        Norm nm{1.0, 1.0, false, false};
        double base_mass_u = 0.0, base_mass_v = 0.0;  // sum of the (unnormalised) weights of the threads before me
        f32x2 x2[E];  // my (u, v) bin pairs (the gradient kernel needs them again at the end)
        (void)base_mass_u;
        (void)base_mass_v;

        // ---- stages 1 + 2: blocked read of my E bins (conflict free: E is odd), masses and CDFs
        //      (fp64 accumulation, one rounding to fp32 per entry) ---------------------------------------
        if constexpr (FROM_BINS) {
            // Pass 1: my E (u, v) bin pairs -> values to accumulate (x, x^2, |z| or |z|^2) and their local
            // sums, in packed fp32.  The per-thread sums T are then scanned across the CTA in fp64.
            const bool inside = in_u && in_v;
            // One-warp CTAs: the entries between the end of a raw row and the end of the last thread's bins are
            // zeroed IN the landing row (one store per thread and row, a warp barrier), so nobody masks what it
            // read.  With one warp per frame the warp of the thread that straddles the row end is the whole frame:
            // the register masks below cost it 33 x (2 ISETP + 2 FSEL) issue slots, 5 % of the kernel.
            constexpr bool ZERO_TAIL = (NW == 1) && !CPLX;
            if constexpr (ZERO_TAIL) {
                for (int idx = n + tid; idx < TPF * E; idx += TPF) sts32(sb + LAND + cur_lead_u + 4u * idx, 0.0f);
                for (int idx = m + tid; idx < TPF * E; idx += TPF) sts32(sb + LAND + LY::LAND_ROW + cur_lead_v + 4u * idx, 0.0f);
                __syncwarp();
            }
#pragma unroll
            for (int c = 0; c < E; ++c) {  // (past the row: zeros, or finite garbage inside the landing rows that is masked)
                if constexpr (CPLX) {  // |z|^2 = re^2 + im^2 directly (no square root), or |z|
                    float re, im;
                    lds64(rawU + 8 * c, re, im);
                    const float s2 = __fmaf_rn(re, re, __fmul_rn(im, im));
                    lds64(rawV + 8 * c, re, im);
                    const float t2 = __fmaf_rn(re, re, __fmul_rn(im, im));
                    x2[c] = pack2(square ? s2 : sqrtf(s2), square ? t2 : sqrtf(t2));
                } else {
                    x2[c] = lds32x2(rawU + 4 * c, rawV + 4 * c);
                }
            }
            if constexpr (!ZERO_TAIL) {
                if (!inside) {
#pragma unroll
                    for (int c = 0; c < E; ++c) x2[c] = mask2(x2[c], e0 + c < n, e0 + c < m);
                }
            }
            (void)inside;
            const bool sq = square && !CPLX;
            // Normalised spectra (every `Wasserstein1D` call) take the packed fp32 route: a few ulp, at a third of the
            // instructions of the fp64 cumsum of raw weights (module-level `wasserstein_1d`, kernel mode MODE_RAW).
            constexpr bool exact = (MODE == MODE_RAW);
            double off_u = 0.0, off_v = 0.0, nxt_u = 0.0, nxt_v = 0.0, tot_u, tot_v;
            if constexpr (exact) {
                raw_cumsum(x2, sq, off_u, off_v, [](int, float) {}, [](int, float) {});
                cta_scan2d<TPF>(off_u, off_v, tot_u, tot_v, scratch, tid);
            } else {
                // the adds of cdf_entries (a segment's sum is its last prefix), written out like the local sums of
                // sot_long.cu: as a call, ptxas allocates the 32 x 33 complex gradient kernel differently
                constexpr int NSEG = cdf_segments(E);
                f32x2 t2 = 0;
#pragma unroll
                for (int s = 0; s < NSEG; ++s) {
                    f32x2 acc2 = 0;
                    if (sq) {
#pragma unroll
                        for (int c = seg_begin<E>(s); c < seg_begin<E>(s + 1); ++c) acc2 = fma2(x2[c], x2[c], acc2);
                    } else {
#pragma unroll
                        for (int c = seg_begin<E>(s); c < seg_begin<E>(s + 1); ++c) acc2 = add2(acc2, x2[c]);
                    }
                    t2 = NSEG == 1 ? acc2 : add2(t2, acc2);
                }
                float Tu, Tv;
                unpack2(t2, Tu, Tv);
                // (the barrier inside also orders the raw reads before the CDF writes)
                cta_scan2<TPF, false, true>(Tu, Tv, off_u, off_v, nxt_u, nxt_v, tot_u, tot_v, scratch, tid);
            }
            base_mass_u = off_u;
            base_mass_v = off_v;
            nm = normalise<exact>(tot_u, tot_v, cut_scale);
            if constexpr (NW == 1) __syncwarp();
            if constexpr (exact) {
                double tu = off_u, tv = off_v;
                raw_cumsum(
                    x2, sq, tu, tv, [&](int c, float x) { if (in_u || e0 + c < n) sts32(A0 + 4 * (e0 + c), x); },
                    [&](int c, float x) { if (in_v || e0 + c < m) sts32(B0 + 4 * (e0 + c), x); });
            } else {
                // Every thread stores all E entries (rows hold TPF * E floats and more): no per-element guards, one
                // code path -- the few threads whose bins straddle or lie past the end of a row used to drag
                // their whole warp through a second, guarded copy of this loop.  What they wrote past the row is
                // overwritten below (sentinels).
                const CdfScale k = cdf_scale(off_u, off_v, nxt_u, nxt_v, nm);
                const auto store_u = [&](int c, float x) { sts32(A0 + 4 * (e0 + c), x); };
                const auto store_v = [&](int c, float x) { sts32(B0 + 4 * (e0 + c), x); };
                if (sq) cdf_entries<true>(x2, k, store_u, store_v); else cdf_entries<false>(x2, k, store_u, store_v);
            }
            // a poisoned frame skips the walk (its +inf sentinels must stay unique) and NaN is written instead
            finite = finite_frame(tot_u, tot_v, nm);
        } else {
            float xu[E], xv[E];
#pragma unroll
            for (int c = 0; c < E; ++c) {
                xu[c] = (e0 + c < n) ? lds32(rawU + 4 * c) : 0.0f;
                xv[c] = (e0 + c < m) ? lds32(rawV + 4 * c) : 0.0f;
                x2[c] = 0;
            }
            cta_sync<TPF>();  // the rows are shifted in place by `lead`: all reads before any write
#pragma unroll
            for (int c = 0; c < E; ++c) {
                if (e0 + c < n) sts32(A0 + 4 * (e0 + c), fminf(xu[c], FLT_BIG));
                if (e0 + c < m) sts32(B0 + 4 * (e0 + c), fminf(xv[c], FLT_BIG));
            }
        }
        // +inf sentinels at [n] / [m]: written by the thread whose bins hold that index, AFTER its own stores
        // (program order), or by thread 0 when no thread's bins reach that far
        if ((e0 <= n && n < e0 + E) || (tid == 0 && n >= TPF * E)) sts32(A0 + 4 * n, f_inf());
        if ((e0 <= m && m < e0 + E) || (tid == 0 && m >= TPF * E)) sts32(B0 + 4 * m, f_inf());
        if constexpr (WITH_GRAD) {
            // the previous frame's output store must have finished READING its staging rows (the dL/dCDF rows)
            // before anybody writes them again (below, in the walk, or in stage 4 of a poisoned frame): thread 0
            // waits for that before it arrives at the barrier.  The store has had two stages to drain.
            if (tid == 0) bulk_wait_read_all();
        }
        cta_sync<TPF>();
        if constexpr (WITH_GRAD && FROM_BINS) {
            // the gradient stage sums dL/dCDF over all E entries of every thread without guards: zero what lies
            // past the end of the rows (the walk only writes real entries).  Spread over the CTA: entry n + tid,
            // normally one store per thread and row (nobody else touches these entries before the barriers that
            // precede the gradient stage).
            for (int idx = n + tid; idx < TPF * E; idx += TPF) sts32o<LY::G_OFF>(A0 + 4 * idx, 0.0f);
            for (int idx = m + tid; idx < TPF * E; idx += TPF) sts32o<LY::G_OFF>(B0 + 4 * idx, 0.0f);
        }
        int cntf[NCH];  // slots of my chunks in THIS frame (sub-warp frames: none when the frame is poisoned)
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) cntf[ch] = cnt[ch];
        uint32_t adrA[NCH], adrB[NCH];
        float a[NCH], pa[NCH], b[NCH], pb[NCH], qprev[NCH];
        int i0[NCH];
#pragma unroll
        for (int ch = 0; ch < NCH; ++ch) {
            adrA[ch] = A0;
            adrB[ch] = B0;
            a[ch] = pa[ch] = b[ch] = pb[ch] = qprev[ch] = 0.0f;
            i0[ch] = 0;
        }
        if (finite) {
            // ---- stage 3a: merge-path partition (fixed-trip, branch-free bit descent) ---------------
            // i0 = number of u entries among the first k0 merged slots (u first on equal values):
            // the largest i in [lo, hi] with A[i-1] <= B[k0-i].  The NCH searches are interleaved.
            uint32_t cur[NCH], hiA[NCH], sumAB[NCH];
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) {
                cur[ch] = A0 + 4u * max(0, k0[ch] - m);  // address of A[i] for the current i
                hiA[ch] = A0 + 4u * min(k0[ch], n);
                sumAB[ch] = A0 + B0 + 4u * k0[ch];  // addr(A[i]) + addr(B[k0-i]) is constant
            }
            search_descent<SEARCH_TOP, NCH>(cur, hiA, sumAB);
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) i0[ch] = static_cast<int>((cur[ch] - A0) >> 2);
#pragma unroll
            for (int ch = 0; ch < NCH; ++ch) {
                adrA[ch] = A0 + 4u * i0[ch];
                adrB[ch] = B0 + 4u * (k0[ch] - i0[ch]);
                a[ch] = lds32(adrA[ch]);
                b[ch] = lds32(adrB[ch]);
                if constexpr (UNI) {  // pa := position difference of the two heads (indices clamped), pb := 0
                    const float xa = pu0 + hstep * static_cast<float>(min(i0[ch], n - 1));
                    const float xb = pv0 + hstep * static_cast<float>(min(k0[ch] - i0[ch], m - 1));
                    pa[ch] = xa - xb;
                    pb[ch] = 0.0f;
                } else {
                    pa[ch] = lds32o<LY::POS_OFF>(adrA[ch]);
                    pb[ch] = lds32o<LY::POS_OFF>(adrB[ch]);
                }
                if (k0[ch] > 0) {  // else: the zero the reference pads in front of qs (losses.py:301)
                    const float al = i0[ch] > 0 ? lds32(adrA[ch] - 4) : -f_inf();
                    const float bl = k0[ch] - i0[ch] > 0 ? lds32(adrB[ch] - 4) : -f_inf();
                    qprev[ch] = fmaxf(al, bl);
                }
            }
        }

        if constexpr (OUT == OUT_LOSS) {
            // ---- stage 3b (forward): walk my slots ---------------------------------------------------
            if (finite) {
                auto fstep = [&](auto CH) {
                    constexpr int ch = decltype(CH)::value;
                    const float q = fminf(a[ch], b[ch]);
                    const float D = UNI ? cost_of_gap<PMODE>(pa[ch], args.p) : transport_cost<PMODE>(pa[ch], pb[ch], args.p);
                    float dq = q - qprev[ch];
                    if constexpr (!NOLIM) {
                        float keep;
                        asm("fma.rn.sat.f32 %0, %1, 0fDD800000, %2;" : "=f"(keep) : "f"(q), "f"(keep_c));  // q * -2^60 + c
                        dq = __fmul_rn(dq, keep);
                    }
                    acc[ch] = fmaf(dq, D, acc[ch]);
                    qprev[ch] = q;
                    uint32_t consumed;
                    if constexpr (UNI)
                        advance_uni(a[ch], pa[ch], b[ch], adrA[ch], adrB[ch], consumed, hstep, -hstep, wk);
                    else
                        advance<POS4>(a[ch], pa[ch], b[ch], pb[ch], adrA[ch], adrB[ch], consumed, wk);
                };
                int s = 0;
                if constexpr (NCH == 2) {
#pragma unroll 2
                    for (; s < cntf[1]; ++s) {
                        fstep(IC<0>{});
                        fstep(IC<1>{});
                    }
                }
#pragma unroll 4
                for (; s < cntf[0]; ++s) fstep(IC<0>{});
            }
        } else if constexpr (OUT == OUT_GRAD) {
            // ---- stage 3b (gradient): walk + dL/dCDF -----------------------------------------------------
            // m*d of a tie group is fixed at its first slot; dL/dCDF is nonzero only at a group's LAST
            // slot: G = (m*d)_group - (m*d)_next group (SURVEY.md 3.3).  It is stored one step later,
            // when the next slot is known.  (It cannot overwrite the consumed CDF entry or its position:
            // a slower thread may still load that entry as the head that ends its own range.)
            if constexpr (SUB) {
                // the frames of a warp may differ in `finite`, and the block below contains warp barriers: a
                // poisoned frame goes through it with empty chunks (no slot is walked, nothing is stored)
                if (!finite) {
#pragma unroll
                    for (int ch = 0; ch < NCH; ++ch) cntf[ch] = 0;
                }
            }
            if (SUB || finite) {
                float md_prev[NCH];
                bool inherited[NCH];  // the open group started before my chunk: its m*d is not known yet
                uint32_t consumed[NCH], fix[NCH];
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    const float q = fminf(a[ch], b[ch]);
                    const float D = UNI ? cost_of_gap<PMODE>(pa[ch], args.p) : transport_cost<PMODE>(pa[ch], pb[ch], args.p);
                    const float fm = (q > thr) ? 0.0f : D;
                    inherited[ch] = (k0[ch] > 0) && (q == qprev[ch]);
                    md_prev[ch] = inherited[ch] ? 0.0f : fm;
                    float dq = q - qprev[ch];
                    dq = (q > thr) ? 0.0f : dq;
                    if (cntf[ch] > 0) {
                        acc[ch] = fmaf(dq, D, acc[ch]);
                        qprev[ch] = q;
                    }
                    consumed[ch] = 0;
                    fix[ch] = NO_FIX;
                }
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch)
                    if (cntf[ch] > 0) {
                        if constexpr (UNI)
                            advance_uni(a[ch], pa[ch], b[ch], adrA[ch], adrB[ch], consumed[ch], hstep, -hstep, wk);
                        else
                            advance<POS4>(a[ch], pa[ch], b[ch], pb[ch], adrA[ch], adrB[ch], consumed[ch], wk);
                    }
                auto gstep = [&](auto CH) {
                    constexpr int ch = decltype(CH)::value;
                    const float q = fminf(a[ch], b[ch]);
                    const float D = UNI ? cost_of_gap<PMODE>(pa[ch], args.p) : transport_cost<PMODE>(pa[ch], pb[ch], args.p);
                    float fmd = D;  // m * d of a group that starts here
                    if constexpr (!NOLIM) {
                        float keep;  // 1 for q <= thr, 0 above (fma pipe, see keep_c)
                        asm("fma.rn.sat.f32 %0, %1, 0fDD800000, %2;" : "=f"(keep) : "f"(q), "f"(keep_c));
                        fmd = __fmul_rn(D, keep);
                    }
                    acc[ch] = fmaf(q - qprev[ch], fmd, acc[ch]);
                    // tie_step(), written out here and below: as a call, ptxas allocates the gradient kernels differently
                    const bool same = (q == qprev[ch]);
                    const float md = same ? md_prev[ch] : fmd;
                    sts32o<LY::G_OFF>(consumed[ch], md_prev[ch] - md);  // dL/dCDF of the previous slot (0 inside a group)
                    fix[ch] = (inherited[ch] && !same) ? consumed[ch] : fix[ch];
                    inherited[ch] = inherited[ch] && same;
                    md_prev[ch] = md;
                    qprev[ch] = q;
                    if constexpr (UNI)
                        advance_uni(a[ch], pa[ch], b[ch], adrA[ch], adrB[ch], consumed[ch], hstep, -hstep, wk);
                    else
                        advance<POS4>(a[ch], pa[ch], b[ch], pb[ch], adrA[ch], adrB[ch], consumed[ch], wk);
                };
                int s = 1;
                if constexpr (NCH == 2) {
#pragma unroll 2
                    for (; s < cntf[1]; ++s) {
                        gstep(IC<0>{});
                        gstep(IC<1>{});
                    }
                }
#pragma unroll 4
                for (; s < cntf[0]; ++s) gstep(IC<0>{});
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    float carry_out = -1.0f;  // -1 = "my whole chunk continues a group opened before it"
                    if (cntf[ch] > 0) {
                        // The slot after my chunk = the first slot of the next chunk (or the virtual slot K: both
                        // heads are the +inf sentinels, a new group with m*d = 0): my heads after the last advance
                        // ARE that slot -- the same shared-memory entries and the same position difference the
                        // next chunk starts from, so no mailbox between the chunks (and no barrier for it).
                        const float qn = fminf(a[ch], b[ch]);
                        const float Dn = UNI ? cost_of_gap<PMODE>(pa[ch], args.p) : transport_cost<PMODE>(pa[ch], pb[ch], args.p);
                        const float mdn = (qn > thr) ? 0.0f : Dn;
                        // tie_step() written out (see gstep), without the update of md_prev: the carry is the m*d of
                        // my last group
                        const bool same = (qn == qprev[ch]);
                        const float md = same ? md_prev[ch] : mdn;
                        sts32o<LY::G_OFF>(consumed[ch], md_prev[ch] - md);
                        fix[ch] = (inherited[ch] && !same) ? consumed[ch] : fix[ch];
                        inherited[ch] = inherited[ch] && same;
                        carry_out = inherited[ch] ? -1.0f : md_prev[ch];
                    }
                    sts32(carry + 4u * (NCH * tid + ch), carry_out);
                }
                // look-back: add the m*d of a tie group that was opened by an earlier chunk
                cta_sync<TPF>();
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    if (fix[ch] != NO_FIX) {
                        const float c = look_back(carry + 4u * (NCH * tid + ch - 1), 4u, lds32);
                        sts32o<LY::G_OFF>(fix[ch], lds32o<LY::G_OFF>(fix[ch]) + c);
                    }
                }
                cta_sync<TPF>();
            }
        } else {
            // ---- stage 3b (plan): emit qs, lower-bound indices, quantile positions, loss ------------------
            // Same partition and tie-group rule; the per-group payload is the pair of lower-bound indices
            // (#{cu < q}, #{cv < q}) -- what `searchsorted(cu, qs)` / `searchsorted(cv, qs)` return
            // (losses.py:219).
            if (finite) {
                int n_inherited[NCH];
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    int i = i0[ch], j = k0[ch] - i0[ch], is = 0, js = 0;
                    bool inherited = (k0[ch] != 0);
                    n_inherited[ch] = 0;
                    for (int s = 0; s < cntf[ch]; ++s) {
                        const float q = fminf(a[ch], b[ch]);
                        const bool take_v = b[ch] < a[ch];
                        if (q != qprev[ch]) {
                            is = i;
                            js = j;
                            inherited = false;
                        }
                        if (inherited) ++n_inherited[ch];
                        const long long o = frame * K + k0[ch] + s;
                        if (args.plan_qs != nullptr) args.plan_qs[o] = q;
                        if (args.plan_iu != nullptr) args.plan_iu[o] = is;
                        if (args.plan_iv != nullptr) args.plan_iv[o] = js;
                        if (args.plan_uq != nullptr) args.plan_uq[o] = lds32(A0 + LY::POS_OFF + 4u * is);
                        if (args.plan_vq != nullptr) args.plan_vq[o] = lds32(B0 + LY::POS_OFF + 4u * js);
                        float dq = q - qprev[ch];
                        dq = (q > thr) ? 0.0f : dq;
                        acc[ch] = fmaf(dq, transport_cost<PMODE>(pa[ch], pb[ch], args.p), acc[ch]);
                        qprev[ch] = q;
                        if (take_v) ++j; else ++i;
                        uint32_t consumed;
                        advance<POS4>(a[ch], pa[ch], b[ch], pb[ch], adrA[ch], adrB[ch], consumed, wk);
                    }
                    sts32(carry + 4u * (NCH * tid + ch),
                          __int_as_float((cntf[ch] == 0 || inherited) ? -1 : ((is << 16) | js)));
                }
                cta_sync<TPF>();
#pragma unroll
                for (int ch = 0; ch < NCH; ++ch) {
                    if (n_inherited[ch] > 0) {
                        const int c = look_back(carry + 4u * (NCH * tid + ch - 1), 4u,
                                                [](uint32_t a) { return __float_as_int(lds32(a)); });
                        const int is2 = c >> 16, js2 = c & 0xffff;
                        for (int t = 0; t < n_inherited[ch]; ++t) {
                            const long long o = frame * K + k0[ch] + t;
                            if (args.plan_iu != nullptr) args.plan_iu[o] = is2;
                            if (args.plan_iv != nullptr) args.plan_iv[o] = js2;
                            if (args.plan_uq != nullptr) args.plan_uq[o] = lds32(A0 + LY::POS_OFF + 4u * is2);
                            if (args.plan_vq != nullptr) args.plan_vq[o] = lds32(B0 + LY::POS_OFF + 4u * js2);
                        }
                    }
                }
                if (args.plan_cu != nullptr)
                    for (int e = tid; e < n; e += TPF) args.plan_cu[frame * n + e] = lds32(A0 + 4u * e);
                if (args.plan_cv != nullptr)
                    for (int e = tid; e < m; e += TPF) args.plan_cv[frame * m + e] = lds32(B0 + 4u * e);
            }
        }

        // ---- loss of the frame: fp32 partials, summed in fp64 ---------------------------------------
        // (gradient kernel from spectra: the cross-warp half of this reduction shares ONE barrier with the suffix
        // scan and the mass-term sums of stage 4, see below)
        constexpr bool MERGED = WITH_GRAD && FROM_BINS;
        double part = 0.0;
        auto reduce_loss_in_warp = [&]() {
            part = static_cast<double>(NCH == 2 ? acc[0] + acc[NCH - 1] : acc[0]);
#pragma unroll
            for (int off = WG / 2; off > 0; off >>= 1) part += __shfl_xor_sync(FULL_MASK, part, off);
        };
        auto write_loss = [&]() {
            if (tid == 0) {
                const float frame_loss = finite ? static_cast<float>(part) : f_nan();
                if (args.loss != nullptr) args.loss[frame] = frame_loss;
                if (active) cta_loss += static_cast<double>(frame_loss);
            }
        };
        if constexpr (!MERGED) {
            reduce_loss_in_warp();
            if constexpr (NW > 1) {
                if ((tid & 31) == 0) scratch[2 * NW + (tid >> 5)] = part;
                __syncthreads();  // (forward / plan: also "every thread is done with the CDF rows")
                part = 0.0;
#pragma unroll
                for (int k = 0; k < NW; ++k) part += scratch[2 * NW + k];
            } else {
                __syncwarp();
            }
            write_loss();
        }

        if constexpr (!WITH_GRAD) {
            // the landing zone (CDF rows) is free: fetch the next frame
            if (elected && has_next && bulk_in) issue_load(fbase + fstride);
        } else {
            // ---- stages 4 + 5: gradient rows, written over the dL/dCDF rows at the phase (address mod 16)
            // of their destination so that the aligned middle can leave by bulk store --------------------
            float* const ou = args.grad_u != nullptr ? args.grad_u + frame * wu : nullptr;
            float* const ov = args.grad_v != nullptr ? args.grad_v + frame * wv : nullptr;
            const uint32_t lead_u = static_cast<uint32_t>(reinterpret_cast<uintptr_t>(ou) & 15);
            const uint32_t lead_v = static_cast<uint32_t>(reinterpret_cast<uintptr_t>(ov) & 15);
            const uint32_t GA0 = A0 + LY::G_OFF, GB0 = B0 + LY::G_OFF;
            // staging rows of the output: the dL/dCDF rows, or (complex) the landing rows, rewritten in place
            constexpr uint32_t STAGE_U = CPLX ? LY::LAND : LY::A + LY::G_OFF;
            constexpr uint32_t STAGE_V = CPLX ? LY::LAND + LY::LAND_ROW : LY::B + LY::G_OFF;
            if constexpr (FROM_BINS) {
                // cumsum transpose: gw_i = sum_{l >= i} dL/dc_l = (sum of the threads after me) + local suffix sum
                // ls_i, and the normalisation chain rule, whose mass term is  sum_i gw_i w_i  -- the sum the
                // reference's autograd forms (w = x^2 / M, losses.py:176-184).  Per thread
                //     sum_i gw_i w_i = off * (T / M) + sum_i ls_i w_i,
                // and over the CTA  sum_t off_t T_t = sum_t S_t P_t  (S_t = my sum of dL/dc, P_t = the sum of the
                // T before me = the base of my CDF entries, kept from stage 2): every term is thread local, so ONE
                // barrier carries the suffix scan, these sums and the loss.  Nothing is read back from the CDF rows
                // (their past-the-end entries are +inf) and their shared-memory traffic is gone.
                // (packed fp32 on (u, v) pairs, like the CDF stage)
                // Real rows: the E local suffix sums are NOT kept (34 registers across the scan): the emit loop below
                // reads dL/dCDF a second time and rebuilds them in the same order -- bit-identical values, +E shared-
                // memory loads per thread, and the register file holds 10 instead of 8 frames per SM.  The first
                // three pairs stay in registers: the emit loop of the thread before me writes its last outputs over
                // them (output staging is in place, shifted by the destination's 16-byte phase of <= 3 floats).
                constexpr bool KEEP_LS = CPLX;
                constexpr int NKEEP = (E < 3) ? E : 3;
                f32x2 ls2[KEEP_LS ? E : 1];
                f32x2 gk[NKEEP];
                f32x2 s2 = 0, d2 = 0;
                const bool sqw = square && !CPLX;  // x2 holds magnitudes: w ~ x^2; else x2 is what was accumulated
                auto suffix_pass = [&](auto SQW) {
#pragma unroll
                    for (int c = E - 1; c >= 0; --c) {
                        const f32x2 g2 = lds32x2(GA0 + 4 * (e0 + c), GB0 + 4 * (e0 + c));
                        s2 = add2(s2, g2);
                        if constexpr (KEEP_LS) ls2[c] = s2;
                        if (c < NKEEP) gk[c] = g2;
                        d2 = fma2(decltype(SQW)::value ? mul2(x2[c], x2[c]) : x2[c], s2, d2);
                    }
                };
                if (sqw) suffix_pass(std::true_type{}); else suffix_pass(std::false_type{});
                (void)ls2;
                float su, sv, du, dv;
                unpack2(s2, su, sv);
                unpack2(d2, du, dv);
                // my share of sum_i gw_i w_i (the factor 1/M is applied once, below: inv_u / inv_v)
                reduce_loss_in_warp();
                double dot_u = static_cast<double>(su) * base_mass_u + static_cast<double>(du);
                double dot_v = static_cast<double>(sv) * base_mass_v + static_cast<double>(dv);
#pragma unroll
                for (int off = WG / 2; off > 0; off >>= 1) {
                    dot_u += __shfl_xor_sync(FULL_MASK, dot_u, off);
                    dot_v += __shfl_xor_sync(FULL_MASK, dot_v, off);
                }
                if constexpr (NW > 1) {
                    if ((tid & 31) == 0) {
                        scratch[2 * NW + (tid >> 5)] = part;
                        scratch[6 * NW + (tid >> 5)] = dot_u;
                        scratch[7 * NW + (tid >> 5)] = dot_v;
                    }
                }
                double off_u, off_v, nu_ = 0.0, nv_ = 0.0, tu, tv;
                cta_scan2<TPF, true, false>(su, sv, off_u, off_v, nu_, nv_, tu, tv, scratch + 4 * NW, tid);  // (barrier)
                (void)nu_;
                (void)nv_;
                if constexpr (NW > 1) {
                    part = 0.0;
                    dot_u = 0.0;
                    dot_v = 0.0;
#pragma unroll
                    for (int k = 0; k < NW; ++k) {
                        part += scratch[2 * NW + k];
                        dot_u += scratch[6 * NW + k];
                        dot_v += scratch[7 * NW + k];
                    }
                } else {
                    __syncwarp();
                }
                write_loss();
                dot_u *= nm.inv_u;
                dot_v *= nm.inv_v;
                // every thread has read its dL/dCDF entries and is done with the CDF rows (barrier above): the CDF
                // rows can take the next frame, the dL/dCDF rows the finished gradients
                if constexpr (!CPLX) {  // (complex: the landing rows are the output staging, see below)
                    if (elected && has_next && bulk_in) issue_load(fbase + fstride);
                }
                double corr_u, corr_v;
                mass_terms(nm, cut_scale, dot_u, dot_v, corr_u, corr_v);
                // gw = offset + local suffix; (offset - corr) is formed in fp64 before rounding
                const float bu = static_cast<float>(off_u - corr_u), bv = static_cast<float>(off_v - corr_v);
                float ku, kv;
                grad_scale(nm, upstream_of(args, frame), square, finite, ku, kv);
                if constexpr (!CPLX) {
                    const f32x2 b2 = pack2(bu, bv), k2 = pack2(ku, kv);
                    const uint32_t out_u = GA0 + lead_u + 4 * e0, out_v = GB0 + lead_v + 4 * e0;
                    // (uniform choice hoisted out of the element loop; all E entries are stored: what lies past the
                    // row stays in the staging row)
                    auto emit = [&](auto SQ) {
                        f32x2 r2 = 0;  // the local suffix sums again, same order as above
#pragma unroll
                        for (int c = E - 1; c >= 0; --c) {  // (descending: what I overwrite I have read)
                            r2 = add2(r2, c < NKEEP ? gk[c] : lds32x2(GA0 + 4 * (e0 + c), GB0 + 4 * (e0 + c)));
                            f32x2 g2 = mul2(add2(b2, r2), k2);
                            if constexpr (decltype(SQ)::value) g2 = mul2(g2, x2[c]);
                            float ga, gb;
                            unpack2(g2, ga, gb);
                            sts32(out_u + 4 * c, ga);
                            sts32(out_v + 4 * c, gb);
                        }
                    };
                    if (square) emit(std::true_type{}); else emit(std::false_type{});
                } else {
                    // d|z|^2/dz = 2z, d|z|/dz = z/|z| (0 at 0, like torch.abs): dL/dz = f * z, written over z.
                    // One row at a time; if the destination's phase differs from the source's the row moves
                    // by 8 bytes inside the landing row, so everybody reads before anybody writes.
                    float lsu[E], lsv[E];
#pragma unroll
                    for (int c = 0; c < E; ++c) unpack2(ls2[c], lsu[c], lsv[c]);
                    auto finish_row = [&](uint32_t raw, uint32_t stage, uint32_t lead_src, uint32_t lead_dst,
                                          const float (&ls)[E], float base, float k, int width) {
                        float re[E], im[E];
#pragma unroll
                        for (int c = 0; c < E; ++c) lds64(raw + 8 * c, re[c], im[c]);
                        if (lead_src != lead_dst) cta_sync<TPF>();
#pragma unroll
                        for (int c = 0; c < E; ++c) {
                            float f = (base + ls[c]) * k;
                            if (!square) {
                                const float mag = sqrtf(__fmaf_rn(re[c], re[c], __fmul_rn(im[c], im[c])));
                                f = mag > 0.0f ? f / mag : f;  // z = 0: the gradient is 0 (torch.abs), NaN stays NaN
                            }
                            if (e0 + c < width) sts64(sb + stage + lead_dst + 8 * (e0 + c), f * re[c], f * im[c]);
                        }
                    };
                    finish_row(rawU, STAGE_U, cur_lead_u, lead_u, lsu, bu, ku, n);
                    finish_row(rawV, STAGE_V, cur_lead_v, lead_v, lsv, bv, kv, m);
                }
            } else {
                // parity harness: the rows ARE dL/dCDF, only shifted to the destination's phase
                float og_u[E], og_v[E];
#pragma unroll
                for (int c = 0; c < E; ++c) {
                    og_u[c] = (e0 + c < n) ? lds32(GA0 + 4 * (e0 + c)) : 0.0f;
                    og_v[c] = (e0 + c < m) ? lds32(GB0 + 4 * (e0 + c)) : 0.0f;
                }
                cta_sync<TPF>();
                if (elected && has_next && bulk_in) issue_load(fbase + fstride);
#pragma unroll
                for (int c = 0; c < E; ++c) {
                    if (e0 + c < n) sts32(GA0 + lead_u + 4 * (e0 + c), og_u[c]);
                    if (e0 + c < m) sts32(GB0 + lead_v + 4 * (e0 + c), og_v[c]);
                }
            }
            fence_async_smem();  // my generic-proxy writes, before the bulk store reads them
            cta_sync<TPF>();
            // aligned middle by bulk store, the (< 4)-float edges by plain stores
            {
                const uint32_t head_u = min((16u - lead_u) & 15u, 4u * wu);  // bytes before the aligned middle
                const uint32_t head_v = min((16u - lead_v) & 15u, 4u * wv);
                const uint32_t body_u = (4u * wu - head_u) & ~15u, body_v = (4u * wv - head_v) & ~15u;
                if (tid == 0) {
                    if (ou != nullptr && body_u > 0)
                        bulk_s2g(reinterpret_cast<char*>(ou) + head_u, smem + STAGE_U + lead_u + head_u, body_u);
                    if (ov != nullptr && body_v > 0)
                        bulk_s2g(reinterpret_cast<char*>(ov) + head_v, smem + STAGE_V + lead_v + head_v, body_v);
                    bulk_commit();
                }
                if (tid < 8 && ou != nullptr) {  // threads 0-3: head floats, 4-7: tail floats
                    const int hf = static_cast<int>(head_u >> 2), tf = wu - hf - static_cast<int>(body_u >> 2);
                    const int idx = tid < 4 ? tid : wu - tf + (tid - 4);
                    if (tid < 4 ? (tid < hf) : (tid - 4 < tf)) ou[idx] = lds32(sb + STAGE_U + lead_u + 4u * idx);
                }
                if (tid >= 8 && tid < 16 && ov != nullptr) {
                    const int t8 = tid - 8;
                    const int hf = static_cast<int>(head_v >> 2), tf = wv - hf - static_cast<int>(body_v >> 2);
                    const int idx = t8 < 4 ? t8 : wv - tf + (t8 - 4);
                    if (t8 < 4 ? (t8 < hf) : (t8 - 4 < tf)) ov[idx] = lds32(sb + STAGE_V + lead_v + 4u * idx);
                }
                if constexpr (CPLX) {
                    // the landing rows double as output staging: the next frame may only land once the bulk
                    // store has read them (and the edge stores, program order of threads 0-15, are done)
                    cta_sync<TPF>();
                    if (tid == 0) {
                        bulk_wait_read_all();
                        if (has_next && bulk_in) issue_load(fbase + fstride);
                    }
                }
            }
        }
    }
    if constexpr (SUB) {  // the frames of the warp kept their own sums (lane 0 of each group): fold them into lane 0
#pragma unroll
        for (int g = 1; g < FPW; ++g) {
            const double other = __shfl_sync(FULL_MASK, cta_loss, g * TPF);
            if (threadIdx.x == 0) cta_loss += other;
        }
    }
    if (threadIdx.x == 0 && args.loss_sum != nullptr) add_cta_loss(args, cta_loss);  // one atomic per CTA
    if constexpr (WITH_GRAD) {
        if (tid == 0) bulk_wait_read_all();  // shared memory must outlive the last bulk store
    }
}

}  // namespace sot
