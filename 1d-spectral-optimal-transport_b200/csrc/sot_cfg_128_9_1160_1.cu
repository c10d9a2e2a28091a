// Kernel instantiations: 128 threads per frame, 9 bins per thread, shared-memory rows of 1160 floats,
// 1 merge chain(s) per thread.
#include "sot_launch.cuh"
SOT_DEFINE_CONFIG(128, 9, 1160, 1, 1)
