// Line lengths (rows W and columns H) the pass kernels are instantiated for.  A length L must be
// E*m*E with E = 16 (where L/256 is a valid middle) or 8, m 5-smooth with a power-of-two part of at most 16,
// and L/E a multiple of 8 (fft_tile.cuh: FftPlan).
// 768 = 16*3*16 is the SLM height of the reference (constants.py:6).  1152 = 8*18*8, 1280 = 16*5*16 and
// 1920 = 8*30*8 serve the common 1920x1152 and 1280x1024 panels.  8192 and 16384 use E = 32 and are
// row-only (slab-decomposed transform of one very large plane).
#pragma once
#ifndef SLM_LINE_LENGTHS      // tuning builds pass a shorter list on the command line
#define SLM_LINE_LENGTHS(X) X(64) X(128) X(192) X(256) X(512) X(768) X(1024) X(1152) X(1280) X(1920) X(2048) X(4096) X(8192) X(16384)
#endif
