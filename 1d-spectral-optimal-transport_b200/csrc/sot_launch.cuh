// Per-configuration launcher: one translation unit per configuration of sot_configs.cuh (csrc/sot_cfg_*.cu) so the
// configurations compile in parallel.  Each exposes `sot_launch_<TPF>_<E>_<RS>_<NCH>(request, stream)`; NCH = merge
// chains per thread.
//   TPF threads per frame, E (odd) consecutive bins per thread, RS floats per shared-memory row, FPW frames per CTA;
//   the configuration accepts rows of up to min(TPF * E, RS - 7) bins.
#pragma once
#include <atomic>

#include "sot_kernels.cuh"

namespace sot {

struct LaunchRequest {
    FrameArgs args;
    int out;   // OUT_LOSS / OUT_GRAD / OUT_PLAN
    int mode;  // MODE_SPECTRA / MODE_CDF
};

// rows longer than shared memory holds (sot_long.cu)
cudaError_t sot_launch_long(const LaunchRequest& r, cudaStream_t stream);

// One kernel's resident CTAs per device ordinal, 0 = not set up yet.
using ResidentCache = std::atomic<int>[64];

// CTAs of `kernel` the device holds at once (occupancy x SM count): the grid of a persistent launch, cached in `cache`.
// The forward is launched from the caller's thread, the backward from the autograd engine's thread of that device,
// and one process may drive several devices.  Two threads that both find the slot empty both run `setup` and the
// (idempotent) queries, and store the same value.
template <typename Kernel, typename Setup>
cudaError_t resident_ctas(ResidentCache& cache, Kernel kernel, int threads, int smem_bytes, Setup setup, int& ctas) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const bool cached = dev >= 0 && dev < static_cast<int>(sizeof(cache) / sizeof(cache[0]));
    ctas = cached ? cache[dev].load(std::memory_order_acquire) : 0;
    if (ctas != 0) return cudaSuccess;
    e = setup();
    if (e != cudaSuccess) return e;
    int per_sm = 0, sms = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, smem_bytes);
    if (e != cudaSuccess) return e;
    e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (e != cudaSuccess) return e;
    ctas = (per_sm < 1 ? 1 : per_sm) * sms;
    if (cached) cache[dev].store(ctas, std::memory_order_release);
    return cudaSuccess;
}

template <int TPF, int E, int RS, int NCH, bool UNI, bool CPLX, int PMODE, int OUT, int MODE, int FPW>
cudaError_t launch_one(const FrameArgs& a, cudaStream_t stream) {
    auto kernel = sot_frame_kernel<TPF, E, RS, NCH, UNI, CPLX, PMODE, OUT, MODE, FPW>;
    constexpr int smem_bytes = static_cast<int>(FPW == 1 ? Layout<TPF, RS, OUT, NCH, UNI, CPLX>::TOTAL
                                                         : FPW * Layout<TPF, RS, OUT, NCH, UNI, CPLX>::SLOT);
    static ResidentCache resident;
    int resident_grid = 0;
    const cudaError_t e = resident_ctas(
        resident, kernel, TPF * FPW, smem_bytes,
        [&] { return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes); },
        resident_grid);
    if (e != cudaSuccess) return e;
    const long long ctas = (a.n_frames + FPW - 1) / FPW;  // FPW frames per CTA and iteration
    const unsigned grid = static_cast<unsigned>(ctas < resident_grid ? ctas : resident_grid);
    kernel<<<grid, TPF * FPW, smem_bytes, stream>>>(a);
    return cudaGetLastError();
}

// The sot_frame_kernel instantiation a request needs, by the template arguments that follow the configuration's own.
constexpr int kernel_key(bool uni, bool cplx, int pmode, int out, int mode) {
    return (((mode * 3 + out) * 4 + pmode) * 2 + cplx) * 2 + uni;
}

// Reads the request once and launches the matching kernel of the configuration.  The cases below are every
// instantiation the configuration has.
template <int TPF, int E, int RS, int NCH, int FPW>
cudaError_t launch_config(const LaunchRequest& r, cudaStream_t stream) {
    const FrameArgs& a = r.args;
    // weights used as given (module-level `wasserstein_1d`) and the plan emitter read positions: general grid, any p
    const bool raw = r.mode == MODE_SPECTRA && (a.flags & FLAG_RAW);
    const bool general = raw || r.out == OUT_PLAN;
    const bool uni = !general && (a.flags & FLAG_UNIFORM) && a.pos_u_stride == 0 && a.pos_v_stride == 0 && a.n >= 2;
    const bool spectra = !general && r.mode == MODE_SPECTRA;
    const bool cplx = spectra && (a.flags & FLAG_COMPLEX);  // interleaved complex64 STFT rows in, complex gradients out
    // PMODE 2: p = 2.  PMODE 3: p = 2 on a uniform grid without the cutoff, the walk without its per-slot mask.
    const int pmode = !(spectra && a.p == 2.0f) ? 0 : (uni && !cplx && !(a.flags & FLAG_LIMIT)) ? 3 : 2;
    const int key = kernel_key(uni, cplx, pmode, r.out, raw ? MODE_RAW : r.mode);
#define SOT_KERNEL(U, C, P, O, M) \
    case kernel_key(U, C, P, O, M): return launch_one<TPF, E, RS, NCH, U, C, P, O, M, FPW>(a, stream);
    switch (key) {  // real spectra, loss and gradients: all that a sub-warp configuration (FPW > 1) serves
        SOT_KERNEL(false, false, 0, OUT_LOSS, MODE_SPECTRA)
        SOT_KERNEL(false, false, 0, OUT_GRAD, MODE_SPECTRA)
        SOT_KERNEL(false, false, 2, OUT_LOSS, MODE_SPECTRA)
        SOT_KERNEL(false, false, 2, OUT_GRAD, MODE_SPECTRA)
        SOT_KERNEL(true, false, 0, OUT_LOSS, MODE_SPECTRA)
        SOT_KERNEL(true, false, 0, OUT_GRAD, MODE_SPECTRA)
        SOT_KERNEL(true, false, 2, OUT_LOSS, MODE_SPECTRA)
        SOT_KERNEL(true, false, 2, OUT_GRAD, MODE_SPECTRA)
        SOT_KERNEL(true, false, 3, OUT_LOSS, MODE_SPECTRA)
        SOT_KERNEL(true, false, 3, OUT_GRAD, MODE_SPECTRA)
    }
    if constexpr (FPW == 1) {
        switch (key) {
            // complex rows
            SOT_KERNEL(false, true, 0, OUT_LOSS, MODE_SPECTRA)
            SOT_KERNEL(false, true, 0, OUT_GRAD, MODE_SPECTRA)
            SOT_KERNEL(false, true, 2, OUT_LOSS, MODE_SPECTRA)
            SOT_KERNEL(false, true, 2, OUT_GRAD, MODE_SPECTRA)
            SOT_KERNEL(true, true, 0, OUT_LOSS, MODE_SPECTRA)
            SOT_KERNEL(true, true, 0, OUT_GRAD, MODE_SPECTRA)
            SOT_KERNEL(true, true, 2, OUT_LOSS, MODE_SPECTRA)
            SOT_KERNEL(true, true, 2, OUT_GRAD, MODE_SPECTRA)
            // injected CDF rows
            SOT_KERNEL(false, false, 0, OUT_LOSS, MODE_CDF)
            SOT_KERNEL(false, false, 0, OUT_GRAD, MODE_CDF)
            SOT_KERNEL(true, false, 0, OUT_LOSS, MODE_CDF)
            SOT_KERNEL(true, false, 0, OUT_GRAD, MODE_CDF)
            // raw weights
            SOT_KERNEL(false, false, 0, OUT_LOSS, MODE_RAW)
            SOT_KERNEL(false, false, 0, OUT_GRAD, MODE_RAW)
            SOT_KERNEL(false, false, 0, OUT_PLAN, MODE_RAW)
            // plans
            SOT_KERNEL(false, false, 0, OUT_PLAN, MODE_SPECTRA)
            SOT_KERNEL(false, false, 0, OUT_PLAN, MODE_CDF)
        }
    }
#undef SOT_KERNEL
    return cudaErrorInvalidValue;  // no kernel of this configuration serves the request (`pick_config` sends none)
}

}  // namespace sot

#define SOT_DEFINE_CONFIG(TPF, E, RS, NCH, FPW)                                                            \
    cudaError_t sot_launch_##TPF##_##E##_##RS##_##NCH(const sot::LaunchRequest& r, cudaStream_t stream) { \
        return sot::launch_config<TPF, E, RS, NCH, FPW>(r, stream);                                        \
    }
