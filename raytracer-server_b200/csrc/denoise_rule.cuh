// denoise_rule.cuh — the edge-aware à-trous filter of the denoiser (rtb_render_denoised, rtb_job_begin_denoised,
// rtb_denoise_image): Dammertz et al. 2010, "Edge-Avoiding À-Trous Wavelet Transform for fast Global Illumination
// Filtering", with the variance-driven luminance edge-stop of SVGF (Schied et al. 2017).
//
// Per-pixel buffers (scan-line order, row 0 = top):
//   colour  float4  demodulated illumination rgb | luminance variance of that illumination
//   ga      float4  albedo rgb | depth (path length to the first non-specular hit)
//   gn      float4  normal xyz (0 for a miss) | object id as int bits (-1 = miss)
// Kept free of device-only code: k_atrous calls atrous_pixel on the GPU and the CPU tests compile it into a host harness.
#pragma once

#include <cuda_runtime.h>

#include <cmath>
#include <cstring>

#include "adaptive_rule.cuh"

namespace rtb {

constexpr int DENOISE_MAX_LEVELS = 8;
constexpr float DN_ALBEDO_FLOOR = 1e-3f;   // demodulation divides by max(albedo, this)
constexpr float DN_EPS_COLOR = 1e-4f;      // luminance edge-stop: |l_p - l_q| / (sigma_color * sqrt(var_p) + this)
constexpr float DN_EPS_DEPTH = 1e-3f;      // depth edge-stop: |z_p - z_q| / (sigma_depth * |grad z_p . (p - q)| + this)

struct DenoiseSigmas {
    float color, normal, depth;
};

__host__ __device__ __forceinline__ int dn_float_as_int(float f) {
#ifdef __CUDA_ARCH__
    return __float_as_int(f);
#else
    int i;
    std::memcpy(&i, &f, 4);
    return i;
#endif
}

// 1-D B3-spline taps for k = -2..2: 1/16, 1/4, 3/8, 1/4, 1/16
__host__ __device__ __forceinline__ float b3_tap(int k) { return k == 0 ? 0.375f : (k == 1 || k == -1 ? 0.25f : 0.0625f); }
// 1-D Gaussian taps of the 3x3 variance prefilter for k = -1..1: 1/4, 1/2, 1/4
__host__ __device__ __forceinline__ float g3_tap(int k) { return k == 0 ? 0.5f : 0.25f; }

__host__ __device__ __forceinline__ float3 albedo_floor(float3 a) {
    return make_float3(fmaxf(a.x, DN_ALBEDO_FLOOR), fmaxf(a.y, DN_ALBEDO_FLOOR), fmaxf(a.z, DN_ALBEDO_FLOOR));
}

// linear colour c with luminance variance var -> illumination c / albedo; the variance scales with 1 / lum(albedo)^2
__host__ __device__ __forceinline__ float4 demodulate(float3 c, float var, float3 albedo) {
    const float3 a = albedo_floor(albedo);
    const float la = lum709(a.x, a.y, a.z);
    return make_float4(c.x / a.x, c.y / a.y, c.z / a.z, var / (la * la));
}

__host__ __device__ __forceinline__ float3 remodulate(float4 illum, float3 albedo) {
    const float3 a = albedo_floor(albedo);
    return make_float3(illum.x * a.x, illum.y * a.y, illum.z * a.z);
}

// Weight of tap q for pixel p, without the B3 factor: 0 across object ids (a hard stop: nothing leaks across object
// boundaries or into misses), else max(0, n_p . n_q)^sigma_normal * exp(-|z_p - z_q| / (sigma_depth * dz + eps)) *
// exp(-|l_p - l_q| / (sigma_color * sd_p + eps)).  dz = |grad z_p . (p - q)| in pixels, sd_p = sqrt of p's prefiltered
// variance.
__host__ __device__ __forceinline__ float edge_weight(int obj_p, int obj_q, float3 n_p, float3 n_q, float z_p, float z_q, float dz,
                                                      float l_p, float l_q, float sd_p, DenoiseSigmas s) {
    if (obj_p != obj_q) return 0.0f;
    const float nd = fmaxf(0.0f, n_p.x * n_q.x + n_p.y * n_q.y + n_p.z * n_q.z);
    const float wn = powf(nd, s.normal);
    const float wz = expf(-fabsf(z_p - z_q) / (s.depth * dz + DN_EPS_DEPTH));
    const float wl = expf(-fabsf(l_p - l_q) / (s.color * sd_p + DN_EPS_COLOR));
    return wn * wz * wl;
}

// One à-trous level at pixel (x, y) with step 2^level: the 5x5 B3 taps at (x + i*step, y + j*step) inside the frame, each
// times edge_weight (the centre tap with weight 1).  The variance that drives the luminance stop is a 3x3 Gaussian of
// `col`'s variance around p (taps inside the frame, renormalised); the depth gradient is the central difference of z
// (one-sided at the border).  Returns (sum w c_q / sum w, sum w^2 var_q / (sum w)^2).
__host__ __device__ inline float4 atrous_pixel(const float4* col, const float4* ga, const float4* gn, int W, int H, int x, int y,
                                               int step, DenoiseSigmas s) {
    const int p = y * W + x;
    const float4 cp = col[p];
    float vsum = 0.0f, gsum = 0.0f;
    for (int j = -1; j <= 1; ++j)
        for (int i = -1; i <= 1; ++i) {
            const int xx = x + i, yy = y + j;
            if (xx < 0 || xx >= W || yy < 0 || yy >= H) continue;
            const float g = g3_tap(i) * g3_tap(j);
            vsum += g * col[yy * W + xx].w;
            gsum += g;
        }
    const float sd_p = sqrtf(fmaxf(vsum / gsum, 0.0f));
    const int xl = x > 0 ? x - 1 : x, xr = x < W - 1 ? x + 1 : x, yu = y > 0 ? y - 1 : y, yd = y < H - 1 ? y + 1 : y;
    const float gx = xr > xl ? (ga[y * W + xr].w - ga[y * W + xl].w) / (float)(xr - xl) : 0.0f;
    const float gy = yd > yu ? (ga[yd * W + x].w - ga[yu * W + x].w) / (float)(yd - yu) : 0.0f;
    const float z_p = ga[p].w;
    const float4 np4 = gn[p];
    const float3 n_p = make_float3(np4.x, np4.y, np4.z);
    const int obj_p = dn_float_as_int(np4.w);
    const float l_p = lum709(cp.x, cp.y, cp.z);
    float wsum = 0.0f, v2 = 0.0f, r = 0.0f, g = 0.0f, b = 0.0f;
    for (int j = -2; j <= 2; ++j)
        for (int i = -2; i <= 2; ++i) {
            const int xx = x + i * step, yy = y + j * step;
            if (xx < 0 || xx >= W || yy < 0 || yy >= H) continue;
            const int q = yy * W + xx;
            const float4 cq = col[q];
            float w = b3_tap(i) * b3_tap(j);
            if (i != 0 || j != 0) {
                const float4 nq4 = gn[q];
                const float dz = fabsf(gx * (float)(i * step) + gy * (float)(j * step));
                w *= edge_weight(obj_p, dn_float_as_int(nq4.w), n_p, make_float3(nq4.x, nq4.y, nq4.z), z_p, ga[q].w, dz, l_p,
                                 lum709(cq.x, cq.y, cq.z), sd_p, s);
            }
            wsum += w;
            r += w * cq.x;
            g += w * cq.y;
            b += w * cq.z;
            v2 += w * w * cq.w;
        }
    const float inv = 1.0f / wsum;   // the centre tap keeps wsum > 0
    return make_float4(r * inv, g * inv, b * inv, v2 * inv * inv);
}

}  // namespace rtb
