// dielectric_rule.cuh — the smooth dielectric interface (brdf 3, "glass"): which side a ray arrives from, Snell's law and
// the exact unpolarised Fresnel reflectance.  DESIGN §3e has the whole contract; k_shade (wavefront.cuh), k_gbuffer
// (denoise.cuh) and the f64 glass oracle (tests/glass_oracle.cpp, restated there) follow it.
//
// Material record (DevMaterial): k.x = ior of the medium (air outside), k.y = orientation sign (+1: the stored normal —
// sphere: outward radial, plane: n, triangle: norm((c-a) x (b-a)) — points out of the medium), color_d = transmission tint.
// Kept free of device-only code: the CPU tests compile it into a host harness.
#pragma once

#include <cmath>

#include "device_types.cuh"

namespace rtb {

// The ray arrives from the outside side: the hit was not flipped (it met the side the stored normal points to) and the
// stored normal points out, or it was flipped and the stored normal points in.
__host__ __device__ __forceinline__ bool dielectric_entering(bool flipped, float orient) { return !flipped != (orient < 0.0f); }

// Fresnel reflectance for cos_i = cos of the angle of incidence (>= 0) and eta = n_i / n_t; cos_t receives the cosine of
// the transmitted angle (0 under total internal reflection, where F = 1).
__host__ __device__ __forceinline__ float dielectric_fresnel(float cos_i, float eta, float& cos_t) {
    const float sin2t = eta * eta * (1.0f - cos_i * cos_i);
    if (sin2t >= 1.0f) {
        cos_t = 0.0f;
        return 1.0f;
    }
    cos_t = sqrtf(1.0f - sin2t);
    const float rs = (eta * cos_i - cos_t) / (eta * cos_i + cos_t);
    const float rp = (cos_i - eta * cos_t) / (cos_i + eta * cos_t);
    return 0.5f * (rs * rs + rp * rp);
}

// One dielectric vertex: dir = true (unit) ray direction, nf = facing normal (dot(dir, nf) <= 0), u = brdf u1 of the vertex.
// Returns the new direction; `refracted` says whether the ray crossed the interface (else it was reflected about nf).
__host__ __device__ __forceinline__ float3 dielectric_scatter(float3 dir, float3 nf, bool flipped, float orient, float ior, float u,
                                                              bool& refracted) {
    const float eta = dielectric_entering(flipped, orient) ? 1.0f / ior : ior;
    const float cos_i = -dot(dir, nf);
    float cos_t;
    const float F = dielectric_fresnel(cos_i, eta, cos_t);
    refracted = !(u < F);
    if (!refracted) return dir + (2.0f * cos_i) * nf;
    return eta * dir + (eta * cos_i - cos_t) * nf;
}

}  // namespace rtb
