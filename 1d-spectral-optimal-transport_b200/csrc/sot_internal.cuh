// Error recording and launch counting behind sot_last_error() and sot_launch_count(), shared by every translation
// unit of the library that validates arguments or launches a kernel (defined in sot_capi.cu; not part of the C ABI).
#pragma once
#include <cuda_runtime.h>

namespace sot {

// Records the printf-style message for sot_last_error() and returns `code`.
int fail(int code, const char* fmt, ...);

// The tail of every kernel launch.  `e` is the launch's error (cudaGetLastError() right after it) or an error of its
// set-up: SOT_OK and one more sot_launch_count(), or "<kernel> launch: <CUDA error>" recorded and the error returned.
int launched(cudaError_t e, const char* kernel);

namespace pairwise {
// The pairwise path's per-row stages over `rows` (>= 1) contiguous rows x[rows][n] of their own (defined in
// sot_pairwise.cu; the barycenters run them too).  launch_row_cdfs writes each row's CDF, normalised by its own mass,
// to cdf[rows][(n + 5) & ~3] and its fp64 mass to mass[rows].  launch_row_grads takes dL/dCDF rows dcdf[rows][n]
// (left in place) and writes dL/dx to grad[rows][n]: suffix sums, the normalisation's chain rule and, with `square`,
// x 2x.
int launch_row_cdfs(const float* x, long long rows, int n, bool square, float* cdf, double* mass, cudaStream_t s);
int launch_row_grads(const float* x, long long rows, int n, bool square, const double* mass, float* dcdf, float* grad,
                     cudaStream_t s);
}  // namespace pairwise

}  // namespace sot
