// Kernel instantiations: SUB-WARP frames for short rows (n_fft 512: 257 bins) -- 16 threads per frame, 17 bins per
// thread, two frames per warp, shared-memory rows of 280 floats, 1 merge chain per thread.
#include "sot_launch.cuh"
SOT_DEFINE_CONFIG(16, 17, 280, 1, 2)
