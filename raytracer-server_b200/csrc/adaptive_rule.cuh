// adaptive_rule.cuh — the per-pixel statistic of adaptive sampling (rtb_render_adaptive, rtb_job_begin_adaptive).
//
// After every pass a pixel contributes ONE batch value: the mean luminance of the samples the pass added, per sub-pixel
// clamped to [0, 1] like the output (k_resolve) and averaged over the 2x2 sub-pixels.  The batch values of the tile's B
// passes are independent estimates of the pixel's mean, so their spread gives the standard error of the final estimate.
// Kept free of device-only code: k_adapt calls it on the GPU and the CPU tests compile it into a host harness.
#pragma once

#include <cuda_runtime.h>

#include <cmath>

namespace rtb {

__host__ __device__ __forceinline__ float clamp01(float x) { return fminf(fmaxf(x, 0.0f), 1.0f); }   // NaN -> 0

// Rec. 709 luminance of linear rgb
__host__ __device__ __forceinline__ float lum709(float r, float g, float b) { return 0.2126f * r + 0.7152f * g + 0.0722f * b; }

// One pass of one pixel.
//   sub[s]   the sub-pixel accumulators: rgb sums over every sample so far; .w = lum709 of the sums after the previous pass
//            (0 before the first).  .w is updated in place.
//   inv_n    1 / (samples per sub-pixel in this pass) = 4 / pass_spp
//   mom      (mean, M2) of the pixel's batch values over the previous passes (Welford), updated in place
//   B        passes of the tile including this one
// Returns the estimated standard error of the pixel's final value in 8-bit output levels, measured after gamma_correct:
// 255 * (min(mu + sigma, 1)^(1/2.2) - mu^(1/2.2)) with mu = clamp01(mean), sigma = sqrt(M2 / (B - 1) / B).
// One batch value has no spread: B < 2 returns +inf.
__host__ __device__ __forceinline__ float adapt_pixel(float4 sub[4], float inv_n, float2& mom, int B) {
    float m = 0.0f;
    for (int s = 0; s < 4; ++s) {
        const float l = lum709(sub[s].x, sub[s].y, sub[s].z);
        m += clamp01((l - sub[s].w) * inv_n);
        sub[s].w = l;
    }
    m *= 0.25f;
    const float delta = m - mom.x;
    mom.x += delta / (float)B;
    mom.y += delta * (m - mom.x);
    if (B < 2) return INFINITY;
    const float mu = clamp01(mom.x);
    const float sigma = sqrtf(fmaxf(mom.y, 0.0f) / (float)(B - 1) / (float)B);
    return 255.0f * (powf(fminf(mu + sigma, 1.0f), 1.0f / 2.2f) - powf(mu, 1.0f / 2.2f));
}

}  // namespace rtb
