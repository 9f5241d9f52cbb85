// Per-pixel statistics of a frame's sums, shared by the adaptive stopping test (adaptive_kernels.cu) and the denoiser
// (denoise_kernels.cu).  Every operation is an explicitly rounded intrinsic: the TUs that include this are compiled with
// --fmad=false and without fast-math, and their numpy models (adaptive.py, denoise.py) repeat the same operations.
#pragma once

#include <cuda_runtime.h>

namespace spcu {

// Unbiased variance of a pixel's luminance samples from its sums after nf samples (R, G, B = rgb_sum, Q = lum_sumsq), and the
// mean luminance m itself:
//   L = (0.2126 R + 0.7152 G) + 0.0722 B;  m = L / n;  d = Q / n - m m;  return v = d > 0 ? d (n / (n - 1)) : 0
// (n >= 2: with n = 1 a positive d gives infinity).
__device__ __forceinline__ float lum_variance(float R, float G, float B, float Q, float nf, float& m)
{
    // luminance() of shade.cuh, one rounding per operation
    const float L = __fadd_rn(__fadd_rn(__fmul_rn(0.2126f, R), __fmul_rn(0.7152f, G)), __fmul_rn(0.0722f, B));
    m             = __fdiv_rn(L, nf);
    const float d = __fsub_rn(__fdiv_rn(Q, nf), __fmul_rn(m, m));
    return d > 0.0f ? __fmul_rn(d, __fdiv_rn(nf, __fsub_rn(nf, 1.0f))) : 0.0f;
}

// Variance of the mean luminance: lum_variance / n.
__device__ __forceinline__ float mean_lum_variance(float R, float G, float B, float Q, float nf, float& m)
{
    return __fdiv_rn(lum_variance(R, G, B, Q, nf, m), nf);
}

} // namespace spcu
