// Kernel instantiations: 128 threads per frame, 17 bins per thread, shared-memory rows of 2184 floats,
// 2 merge chain(s) per thread.
#include "sot_launch.cuh"
SOT_DEFINE_CONFIG(128, 17, 2184, 2, 1)
