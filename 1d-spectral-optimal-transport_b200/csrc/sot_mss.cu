// Multi-scale spectral (MSS) loss term, the companion of the SOT loss in every paper config
// (reference: losses.py:365-425 `MSSLoss`, :7-36 `mean_difference`, utils.py:145-151 `safe_log`,
// features.py:217-237 `compute_mag`): for one FFT size,
//     S = sum_i  mag_w * d(|zt_i|, |zv_i|) + logmag_w * d(safe_log|zt_i|, safe_log|zv_i|),   d = |a-b| or (a-b)^2
// straight from the two COMPLEX spectrograms -- the reference materialises |z| (and its log) per size.
// HBM-bound streaming work: 16 B read per element forward; 16 B read + 8 or 16 B written backward.
// Persistent grid (SMs x 8 CTAs x 256 threads), two complex elements per 128-bit load, fp32 partials per
// thread (a few hundred terms), fp64 across the CTA, ONE fp64 atomic per CTA.
#include <cuda_runtime.h>

#include <cstdint>

#include "../../include/sot_b200.h"
#include "sot_internal.cuh"

namespace sot {

constexpr float MSS_LOG_EPS = 1e-5f;  // utils.py:145: safe_log replaces x <= eps by eps

struct MssArgs {
    const float* zt;   // target spectrogram, interleaved complex64
    const float* zv;   // predicted spectrogram
    long long count;   // complex elements
    float mag_w, logmag_w;
    int l2;            // 0: L1, 1: L2
    float post_scale;  // forward: sum_out += post_scale * S
    double* sum_out;
    const float* scale;  // backward: device scalar dL/dS (multiplied by post_scale)
    float* grad_zt;
    float* grad_zv;
};

__device__ __forceinline__ float mss_term(float tr, float ti, float vr, float vi, float mag_w, float logmag_w, int l2,
                                          float& ft, float& fv) {
    // returns the element's contribution; ft, fv = d(contribution)/d|zt| / |zt| and d/d|zv| / |zv|
    // (so that the complex gradients are ft * zt and fv * zv; 0 where |z| = 0 like torch.abs)
    const float t = sqrtf(fmaf(tr, tr, ti * ti)), v = sqrtf(fmaf(vr, vr, vi * vi));
    float acc = 0.0f, gt = 0.0f, gv = 0.0f;  // gt = d/dt, gv = d/dv
    if (mag_w > 0.0f) {
        const float d = t - v;
        if (l2) {
            acc = fmaf(mag_w, d * d, acc);
            gt += 2.0f * mag_w * d;
            gv -= 2.0f * mag_w * d;
        } else {
            acc = fmaf(mag_w, fabsf(d), acc);
            const float s = d > 0.0f ? mag_w : (d < 0.0f ? -mag_w : 0.0f);
            gt += s;
            gv -= s;
        }
    }
    if (logmag_w > 0.0f) {
        const bool tl = t > MSS_LOG_EPS, vl = v > MSS_LOG_EPS;
        const float lt = logf(tl ? t : MSS_LOG_EPS), lv = logf(vl ? v : MSS_LOG_EPS);
        const float d = lt - lv;
        float s;
        if (l2) {
            acc = fmaf(logmag_w, d * d, acc);
            s = 2.0f * logmag_w * d;
        } else {
            acc = fmaf(logmag_w, fabsf(d), acc);
            s = d > 0.0f ? logmag_w : (d < 0.0f ? -logmag_w : 0.0f);
        }
        if (tl) gt += s / t;  // torch.where picks the constant below eps: no gradient there
        if (vl) gv -= s / v;
    }
    ft = t > 0.0f ? gt / t : 0.0f;
    fv = v > 0.0f ? gv / v : 0.0f;
    return acc;
}

template <bool BACKWARD>
__global__ void __launch_bounds__(256) sot_mss_kernel(const MssArgs a) {
    const long long tid = blockIdx.x * 256LL + threadIdx.x, nthr = gridDim.x * 256LL;
    const long long pairs = a.count >> 1;  // two complex elements per float4
    const float up = BACKWARD ? (a.scale != nullptr ? *a.scale : 1.0f) * a.post_scale : 0.0f;
    const bool vec = ((reinterpret_cast<uintptr_t>(a.zt) | reinterpret_cast<uintptr_t>(a.zv) |
                       reinterpret_cast<uintptr_t>(a.grad_zt) | reinterpret_cast<uintptr_t>(a.grad_zv)) & 15) == 0;
    float acc = 0.0f;
    if (vec) {
        const float4* t4 = reinterpret_cast<const float4*>(a.zt);
        const float4* v4 = reinterpret_cast<const float4*>(a.zv);
        for (long long i = tid; i < pairs; i += nthr) {
            const float4 t = __ldg(t4 + i), v = __ldg(v4 + i);
            float ft0, fv0, ft1, fv1;
            acc += mss_term(t.x, t.y, v.x, v.y, a.mag_w, a.logmag_w, a.l2, ft0, fv0);
            acc += mss_term(t.z, t.w, v.z, v.w, a.mag_w, a.logmag_w, a.l2, ft1, fv1);
            if constexpr (BACKWARD) {
                if (a.grad_zt != nullptr)
                    reinterpret_cast<float4*>(a.grad_zt)[i] =
                        make_float4(up * ft0 * t.x, up * ft0 * t.y, up * ft1 * t.z, up * ft1 * t.w);
                if (a.grad_zv != nullptr)
                    reinterpret_cast<float4*>(a.grad_zv)[i] =
                        make_float4(up * fv0 * v.x, up * fv0 * v.y, up * fv1 * v.z, up * fv1 * v.w);
            }
        }
    }
    // scalar path: everything when the arrays are only 8-byte aligned, else the odd last element
    const float2* t2 = reinterpret_cast<const float2*>(a.zt);
    const float2* v2 = reinterpret_cast<const float2*>(a.zv);
    for (long long i = (vec ? 2 * pairs : 0) + tid; i < a.count; i += nthr) {
        const float2 t = t2[i], v = v2[i];
        float ft, fv;
        acc += mss_term(t.x, t.y, v.x, v.y, a.mag_w, a.logmag_w, a.l2, ft, fv);
        if constexpr (BACKWARD) {
            if (a.grad_zt != nullptr) reinterpret_cast<float2*>(a.grad_zt)[i] = make_float2(up * ft * t.x, up * ft * t.y);
            if (a.grad_zv != nullptr) reinterpret_cast<float2*>(a.grad_zv)[i] = make_float2(up * fv * v.x, up * fv * v.y);
        }
    }
    if constexpr (!BACKWARD) {
        double s = static_cast<double>(acc);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        __shared__ double part[8];
        if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
        __syncthreads();
        if (threadIdx.x == 0) {
            double tot = 0.0;
#pragma unroll
            for (int k = 0; k < 8; ++k) tot += part[k];
            atomicAdd(a.sum_out, tot * static_cast<double>(a.post_scale));
        }
    }
}

int mss_grid(long long count) {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        if (sms <= 0) sms = 148;
    }
    const long long want = (count / 2 + 255) / 256;
    const long long cap = 8LL * sms;
    return static_cast<int>(want < 1 ? 1 : (want < cap ? want : cap));
}

}  // namespace sot

extern "C" {

int sot_mss_forward_device(const float* zt, const float* zv, int64_t count, float mag_weight, float logmag_weight,
                           int32_t loss_type, float post_scale, double* sum_out, void* stream) {
    if (count < 0 || (count > 0 && (zt == nullptr || zv == nullptr)) || sum_out == nullptr)
        return sot::fail(SOT_EINVAL, "sot_mss_forward_device: NULL pointer or negative count");
    if (loss_type != SOT_MSS_L1 && loss_type != SOT_MSS_L2)
        return sot::fail(SOT_EINVAL, "Loss type must be \"L1\" or \"L2\"");
    if (count == 0) return SOT_OK;
    sot::MssArgs a{zt, zv, count, mag_weight, logmag_weight, loss_type == SOT_MSS_L2, post_scale, sum_out, nullptr,
                   nullptr, nullptr};
    sot::sot_mss_kernel<false><<<sot::mss_grid(count), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    return sot::launched(cudaGetLastError(), "sot_mss_kernel");
}

int sot_mss_backward_device(const float* zt, const float* zv, int64_t count, float mag_weight, float logmag_weight,
                            int32_t loss_type, float post_scale, const float* scale, float* grad_zt, float* grad_zv,
                            void* stream) {
    if (count < 0 || (count > 0 && (zt == nullptr || zv == nullptr)))
        return sot::fail(SOT_EINVAL, "sot_mss_backward_device: NULL pointer or negative count");
    if (loss_type != SOT_MSS_L1 && loss_type != SOT_MSS_L2)
        return sot::fail(SOT_EINVAL, "Loss type must be \"L1\" or \"L2\"");
    if (count == 0 || (grad_zt == nullptr && grad_zv == nullptr)) return SOT_OK;
    sot::MssArgs a{zt, zv, count, mag_weight, logmag_weight, loss_type == SOT_MSS_L2, post_scale, nullptr, scale,
                   grad_zt, grad_zv};
    sot::sot_mss_kernel<true><<<sot::mss_grid(count), 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    return sot::launched(cudaGetLastError(), "sot_mss_kernel");
}

}  // extern "C"
