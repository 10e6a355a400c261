// microfacet_rule.cuh — rough metal (brdf 4, "metal"): GGX (Trowbridge-Reitz) microfacet reflection over a conductor with
// Schlick's Fresnel term, and the visible-normal sampler of Heitz 2018 ("Sampling the GGX Distribution of Visible Normals",
// JCGT 7(4)).  DESIGN §3g has the whole contract; k_shade (wavefront.cuh, MODE 6 / 7) and the f64 metal oracle
// (tests/metal_oracle.py, restated there) follow it.
//
// Material record (DevMaterial): k.x = alpha = roughness^2, color_s = F0 (reflectance at normal incidence).
// o = the TRUE direction back to where the ray came from (-d), n = the facing normal, frame = local_coord(n).
// Kept free of device-only code: the CPU tests compile it into a host harness.
#pragma once

#include <cmath>

#include "device_types.cuh"

namespace rtb {

// D(h) = alpha^2 / (pi ((n.h)^2 (alpha^2 - 1) + 1)^2) for c2 = (n.h)^2 and s2 = 1 - (n.h)^2.  The denominator is written
// s2 + alpha^2 c2: with s2 from a cross product it keeps its relative precision where the lobe of a polished metal is narrow.
__host__ __device__ __forceinline__ float metal_D(float a2, float c2, float s2) {
    const float den = s2 + a2 * c2;
    return a2 / (3.14159265358979323846f * den * den);
}

// Smith's Lambda(w) = (sqrt(1 + alpha^2 (1 - c^2) / c^2) - 1) / 2 for c = n.w > 0
__host__ __device__ __forceinline__ float metal_lambda(float a2, float c) {
    const float c2 = c * c;
    return 0.5f * (sqrtf(1.0f + a2 * fmaxf(1.0f - c2, 0.0f) / c2) - 1.0f);
}

// Schlick: F0 + (1 - F0) (1 - o.h)^5, per channel
__host__ __device__ __forceinline__ float3 metal_fresnel(float3 F0, float oh) {
    const float m = fminf(fmaxf(1.0f - oh, 0.0f), 1.0f);
    const float m5 = (m * m) * (m * m) * m;
    return F0 + (f3(1.0f, 1.0f, 1.0f) - F0) * m5;
}

// f(o, i) = F D G2 / (4 (n.o)(n.i)) with the height-correlated G2 = 1 / (1 + Lambda(o) + Lambda(i)); 0 unless both lie above
__host__ __device__ __forceinline__ float3 metal_eval(float3 F0, float alpha, float3 n, float3 o, float3 i) {
    const float no = dot(n, o), ni = dot(n, i);
    if (!(no > 0.0f) || !(ni > 0.0f)) return f3(0.0f, 0.0f, 0.0f);
    const float3 hv = o + i;
    const float inv_h2 = 1.0f / dot(hv, hv);
    const float nh = dot(n, hv);
    const float3 nxh = cross(n, hv);
    const float a2 = alpha * alpha;
    const float D = metal_D(a2, nh * nh * inv_h2, dot(nxh, nxh) * inv_h2);
    const float G2 = 1.0f / (1.0f + metal_lambda(a2, no) + metal_lambda(a2, ni));
    return metal_fresnel(F0, dot(o, hv) * sqrtf(inv_h2)) * (D * G2 / (4.0f * no * ni));
}

// pdf(i) = G1(o) D(h) / (4 n.o), per unit solid angle (0 unless both lie above)
__host__ __device__ __forceinline__ float metal_pdf(float alpha, float3 n, float3 o, float3 i) {
    const float no = dot(n, o), ni = dot(n, i);
    if (!(no > 0.0f) || !(ni > 0.0f)) return 0.0f;
    const float3 hv = o + i;
    const float inv_h2 = 1.0f / dot(hv, hv);
    const float nh = dot(n, hv);
    const float3 nxh = cross(n, hv);
    const float a2 = alpha * alpha;
    return metal_D(a2, nh * nh * inv_h2, dot(nxh, nxh) * inv_h2) / ((1.0f + metal_lambda(a2, no)) * 4.0f * no);
}

// create_local_coord (src/scene.rs:112-123), the frame of the diffuse sampler
__host__ __device__ __forceinline__ void metal_frame(float3 n, float3& u, float3& v) {
    const float3 a = fabsf(n.x) > 0.1f ? f3(0.f, 1.f, 0.f) : f3(1.f, 0.f, 0.f);
    const float3 c = cross(a, n);
    u = c * (1.0f / sqrtf(dot(c, c)));
    v = cross(n, u);
}

// One metal vertex's continuation for brdf u1, u2 of block 0: the visible normal h of Heitz 2018 (isotropic form), i = 2 (o.h) h
// - o, and the weight w = f (n.i) / pdf = F(o.h) G2(o, i) / G1(o).  Returns false (the path ends) if n.o <= 0 or n.i <= 0.
__host__ __device__ __forceinline__ bool metal_sample(float3 F0, float alpha, float3 n, float3 o, float u1, float u2, float3& i, float3& w) {
    float3 tu, tv;
    metal_frame(n, tu, tv);
    const float ox = dot(o, tu), oy = dot(o, tv), oz = dot(o, n);
    // the view direction in the hemisphere configuration (the microsurface stretched to alpha = 1)
    float3 vh = f3(alpha * ox, alpha * oy, oz);
    vh = vh * (1.0f / sqrtf(dot(vh, vh)));
    const float lensq = vh.x * vh.x + vh.y * vh.y;
    const float3 t1 = lensq > 0.0f ? f3(-vh.y, vh.x, 0.0f) * (1.0f / sqrtf(lensq)) : f3(1.0f, 0.0f, 0.0f);
    const float3 t2 = cross(vh, t1);
    // a point of the projected disk: uniform, then squeezed onto the visible half
    const float r = sqrtf(u1);
    float s, c;
#ifdef __CUDA_ARCH__
    sincospif(2.0f * u2, &s, &c);
#else
    s = sinf(6.283185307179586f * u2);
    c = cosf(6.283185307179586f * u2);
#endif
    const float p1 = r * c;
    const float h = 0.5f * (1.0f + vh.z);
    const float p2 = (1.0f - h) * sqrtf(fmaxf(1.0f - p1 * p1, 0.0f)) + h * (r * s);
    const float3 nh = t1 * p1 + t2 * p2 + vh * sqrtf(fmaxf(1.0f - p1 * p1 - p2 * p2, 0.0f));
    // back to the ellipsoid configuration, then into the world frame
    float3 ne = f3(alpha * nh.x, alpha * nh.y, fmaxf(nh.z, 0.0f));
    ne = ne * (1.0f / sqrtf(dot(ne, ne)));
    const float3 hw = tu * ne.x + tv * ne.y + n * ne.z;
    const float oh = dot(o, hw);
    i = (2.0f * oh) * hw - o;
    const float ni = dot(n, i);
    if (!(oz > 0.0f) || !(ni > 0.0f)) return false;
    const float a2 = alpha * alpha;
    const float lo = metal_lambda(a2, oz);
    w = metal_fresnel(F0, oh) * ((1.0f + lo) / (1.0f + lo + metal_lambda(a2, ni)));
    return true;
}

}  // namespace rtb
