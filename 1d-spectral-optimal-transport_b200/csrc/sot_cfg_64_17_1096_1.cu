// Kernel instantiations: 64 threads per frame, 17 bins per thread, shared-memory rows of 1096 floats,
// 1 merge chain(s) per thread.
#include "sot_launch.cuh"
SOT_DEFINE_CONFIG(64, 17, 1096, 1, 1)
