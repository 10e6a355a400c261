// light_rule.cuh — next-event estimation over every emitter (RTB_EST_NEE_ALL_LIGHTS, DESIGN §3f): the choice of a light and
// of a triangle of a mesh light, the uniform point on a triangle and the weight of a light sample.  k_shade (wavefront.cuh,
// MODE 4 / 5) follows it, and so does the f64 oracle of the tests (tests/glass_oracle.cpp, restated there).
//
// The loader (scene_host.cpp) builds the table once per scene in f64 after the transforms: every sphere or mesh whose weight
// w = lum709(max(emitted, 0)) * area is > 0, in object order, chosen with probability p = w / sum w.
// Kept free of device-only code: the CPU tests compile it into a host harness.
#pragma once

#include <cmath>

#include "device_types.cuh"

namespace rtb {

struct DevLight {      // 32 B, one per table entry
    float4 sphere;     // sphere lights: centre | radius
    float pdf_area;    // p / area: the light sample's pdf per unit area
    int32_t obj;       // object index
    int32_t tri_cdf;   // mesh lights: first entry of the mesh's triangle cdf in the cdf table; -1 for a sphere
    int32_t pad;
};

// partition_point(cdf[0, n) <= u), clamped to the last entry: the entry u selects from an inclusive cumulative distribution
__host__ __device__ __forceinline__ int light_pick(const float* cdf, int n, float u) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (cdf[mid] <= u) lo = mid + 1;
        else hi = mid;
    }
    return lo < n ? lo : n - 1;
}

// uniform point of the triangle (a, b, c) for u1, u2 in (0, 1): (1 - sqrt u1) a + sqrt u1 (1 - u2) b + sqrt u1 u2 c
__host__ __device__ __forceinline__ float3 light_tri_point(float3 a, float3 b, float3 c, float u1, float u2) {
    const float s = sqrtf(u1);
    return a * (1.0f - s) + b * (s * (1.0f - u2)) + c * (s * u2);
}

// the triangle's stored normal norm((c - a) x (b - a)); an emitter is two-sided, so its sign does not matter
__host__ __device__ __forceinline__ float3 light_tri_normal(float3 a, float3 b, float3 c) {
    const float3 n = cross(c - a, b - a);
    return n * (1.0f / sqrtf(dot(n, n)));
}

// max(n_f . w, 0) |n_y . w| / (r^2 pdf_area): what multiplies beta Le f for a light point at distance^2 r2 in direction w
// (n_f = the shading point's facing normal, n_y = the light point's normal).  Unlike the reference's estimator, a light
// point behind the shading surface adds nothing, and an emitter shines from both sides.
__host__ __device__ __forceinline__ float light_weight(float3 nf, float3 ny, float3 w, float r2, float pdf_area) {
    return fmaxf(dot(nf, w), 0.0f) * fabsf(dot(ny, w)) / (r2 * pdf_area);
}

}  // namespace rtb
