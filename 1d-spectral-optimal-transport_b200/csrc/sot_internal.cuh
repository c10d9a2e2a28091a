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

}  // namespace sot
