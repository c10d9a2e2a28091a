// The shared-memory kernel configurations, in order of preference: the first one that holds a row serves it (choices
// from measurements on B200, profiles/).  SOT_CONFIG(TPF, E, RS, NCH, FPW): TPF threads per frame, E bins per thread,
// RS floats per shared-memory row, NCH merge chains per thread, FPW frames per CTA.  A configuration holds rows of up
// to min(TPF * E, RS - 7) bins; shared memory per CTA = (4 or 6) * 4 * RS bytes.  Each one's kernels are compiled in
// its own csrc/sot_cfg_*.cu.  No include guard: define SOT_CONFIG, include, undefine.

// <= 272 bins (n_fft 512: 257): two frames per warp, for real spectra with loss or gradient output only
SOT_CONFIG(16, 17, 280, 1, 2)
// <= 288 bins: one warp per frame (plans, CDF harness, raw weights and complex rows of that length)
SOT_CONFIG(32, 9, 296, 1, 1)
// <= 576 bins (n_fft 1024: 513)
SOT_CONFIG(64, 9, 584, 2, 1)
// <= 1056 bins (n_fft 2048: 1025): ONE WARP per frame, 33 bins per thread -- no CTA barriers, half the per-frame
// fixed cost; since the gradient stage rebuilds its suffix sums (162 registers, no spills) 14 % faster than 64 x 17
SOT_CONFIG(32, 33, 1064, 1, 1)
// <= 1088 bins (two warps per frame: the round-1 / early round-2 choice)
SOT_CONFIG(64, 17, 1096, 1, 1)
// <= 1152 bins
SOT_CONFIG(128, 9, 1160, 1, 1)
// <= 2176 bins (n_fft 4096: 2049)
SOT_CONFIG(128, 17, 2184, 2, 1)
// <= 4352 bins (n_fft 8192: 4097)
SOT_CONFIG(256, 17, 4360, 2, 1)
// <= 8448 bins (n_fft 16384: 8193)
SOT_CONFIG(256, 33, 8456, 1, 1)
