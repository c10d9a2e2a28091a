// Kernel instantiations: 256 threads per frame, 33 bins per thread, shared-memory rows of 8456 floats,
// 1 merge chain(s) per thread.
#include "sot_launch.cuh"
SOT_DEFINE_CONFIG(256, 33, 8456, 1, 1)
