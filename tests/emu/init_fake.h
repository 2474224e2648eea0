// tests/emu/init_fake.h -- the intrinsic of csrc/init_kernels.cu that warp_emu.h and cuda_fake.h do not have: the
// round-to-nearest subtraction (no contraction on the CPU either: volatile, as for __dadd_rn).
#pragma once
#include "cuda_fake.h"

inline double __dsub_rn(double a, double b) { volatile double r = a - b; return r; }
