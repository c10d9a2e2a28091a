// Kernel instantiations: 64 threads per frame, 9 bins per thread, shared-memory rows of 584 floats,
// 2 merge chain(s) per thread.
#include "sot_launch.cuh"
SOT_DEFINE_CONFIG(64, 9, 584, 2, 1)
