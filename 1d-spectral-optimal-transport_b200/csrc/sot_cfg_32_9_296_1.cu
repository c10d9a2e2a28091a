// Kernel instantiations: 32 threads per frame, 9 bins per thread, shared-memory rows of 296 floats,
// 1 merge chain(s) per thread.
#include "sot_launch.cuh"
SOT_DEFINE_CONFIG(32, 9, 296, 1, 1)
