// Kernel instantiations: 32 threads per frame, 33 bins per thread, shared-memory rows of 1064 floats,
// 1 merge chain(s) per thread.
#include "sot_launch.cuh"
SOT_DEFINE_CONFIG(32, 33, 1064, 1, 1)
