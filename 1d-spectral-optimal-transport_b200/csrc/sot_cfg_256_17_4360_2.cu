// Kernel instantiations: 256 threads per frame, 17 bins per thread, shared-memory rows of 4360 floats,
// 2 merge chain(s) per thread.
#include "sot_launch.cuh"
SOT_DEFINE_CONFIG(256, 17, 4360, 2, 1)
