// shade.cuh — RNG contract, camera, BRDFs, light sampling: the per-vertex arithmetic of
// Scene::reflected_radiance (reference src/scene.rs:161-244) in fp32.
//
// RNG contract (shared with oracle/rt_oracle.cpp so both consume identical numbers):
//   Philox4x32-10, key = (seed lo, seed hi), counter = (pixel, sample, depth, block),
//   u24(v) = (v + 0.5) * 2^-24 in (0,1) for a 24-bit integer v.
//   pixel  = y_screen * width + x      sample = (sy*2+sx) * (spp/4) + k
//   depth 0 block 0 : tent r1 = u24(x>>8), r2 = u24(y>>8)                          src/server.rs:339-351
//   depth d block 0 : ONE block feeds the whole live vertex (128 bits -> five 24-bit uniforms):
//                     light u1 = u24(x>>8), light u2 = u24(y>>8), russian roulette = u24(z>>8),
//                     brdf u1 = u24(w>>8), brdf u2 = u24((x&255)<<16 | (y&255)<<8 | (z&255))
//           block 1 : phong lobe select = u24(x>>8), light triangle select = u24(y>>8)  (only drawn when needed)
//           block 2 : {brdf u1, u2, lobe} = u24(x>>8, y>>8, z>>8)   dead-MIS "fresh" sample used only for its pdf (:195)
//           block 3 : {light u1, u2, -, select}                      dead-MIS second light point (:206)
//           block 4 : {brdf u1, u2, lobe}                            dead-MIS own BRDF sample (:203)
//   dielectric vertex (DESIGN §3e): block 0 only — russian roulette as for a mirror, reflect iff brdf u1 < Fresnel F;
//                     no light sample, no block 1
//   RTB_EST_NEE_ALL_LIGHTS (DESIGN §3f): block 1 z = light-table entry, block 1 y = triangle of a mesh light, block 0 light
//                     u1, u2 = the point; block 1 is drawn for Phong, more than one light or a mesh light
#pragma once

#include "device_types.cuh"

namespace rtb {

constexpr float PI_F = 3.14159265358979323846f;
constexpr float INV_PI_F = 0.318309886183790671538f;

// The ten round keys (k + i * Weyl constant) are computed once on the host and live in the kernel parameters: after
// unrolling they are constant-bank operands of the XORs, not ten pairs of additions per block.
struct PhiloxKeys {
    uint32_t k0[10], k1[10];
};
__host__ __device__ inline PhiloxKeys philox_keys(uint32_t k0, uint32_t k1) {
    PhiloxKeys K;
    for (int i = 0; i < 10; ++i) {
        K.k0[i] = k0 + (uint32_t)i * 0x9E3779B9u;
        K.k1[i] = k1 + (uint32_t)i * 0xBB67AE85u;
    }
    return K;
}
__device__ __forceinline__ uint4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const PhiloxKeys& K) {
#pragma unroll
    for (int i = 0; i < 10; ++i) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
        uint32_t n0 = hi1 ^ c1 ^ K.k0[i], n2 = hi0 ^ c3 ^ K.k1[i];
        c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    }
    return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float u01(uint32_t x) { return ((float)(x >> 8) + 0.5f) * (1.0f / 16777216.0f); }
__device__ __forceinline__ float u24(uint32_t v) { return ((float)v + 0.5f) * (1.0f / 16777216.0f); }
__device__ __forceinline__ float4 rng_block(uint32_t pixel, uint32_t sample, uint32_t depth, uint32_t block, const PhiloxKeys& K) {
    uint4 r = philox4x32_10(pixel, sample, depth, block, K);
    return make_float4(u01(r.x), u01(r.y), u01(r.z), u01(r.w));
}
// the five uniforms of a live vertex from ONE Philox block (see the contract above)
struct VertexRng {
    float light_u1, light_u2, rr, brdf_u1, brdf_u2;
};
__device__ __forceinline__ VertexRng rng_vertex(uint32_t pixel, uint32_t sample, uint32_t depth, const PhiloxKeys& K) {
    uint4 r = philox4x32_10(pixel, sample, depth, 0u, K);
    VertexRng v;
    v.light_u1 = u24(r.x >> 8);
    v.light_u2 = u24(r.y >> 8);
    v.rr = u24(r.z >> 8);
    v.brdf_u1 = u24(r.w >> 8);
    v.brdf_u2 = u24(((r.x & 0xffu) << 16) | ((r.y & 0xffu) << 8) | (r.z & 0xffu));
    return v;
}

// ---- camera (sample_pixel, src/server.rs:328-357) ---------------------------------------------
struct Camera {
    float3 pos, dir, cx, cy;
    float inv_w, inv_h;
};
__host__ __device__ inline Camera make_camera(const float* cam_pos, const float* cam_dir, int width, int height) {
    Camera c;
    c.pos = f3(cam_pos[0], cam_pos[1], cam_pos[2]);
    c.dir = f3(cam_dir[0], cam_dir[1], cam_dir[2]);
    float w = (float)width, h = (float)height;
    c.cx = f3(w * 0.5135f / h, 0.f, 0.f);
    float3 cr = cross(c.cx, c.dir);
    float len = sqrtf(dot(cr, cr));
    c.cy = f3(cr.x / len * 0.5135f, cr.y / len * 0.5135f, cr.z / len * 0.5135f);
    c.inv_w = 1.0f / w;
    c.inv_h = 1.0f / h;
    return c;
}
__device__ __forceinline__ float tent(float u) {  // src/server.rs:339-344
    float r = 2.0f * u;
    return r < 1.0f ? sqrtf(r) - 1.0f : 1.0f - sqrtf(2.0f - r);
}
// x, y_sampler = bottom-up row (height - y_screen - 1, src/server.rs:181)
__device__ __forceinline__ float3 camera_dir(const Camera& c, int x, int y_sampler, int sx, int sy, float dx, float dy,
                                             float w, float h) {
    float fx = (((float)sx + 0.5f + dx) / 2.0f + (float)x) / w - 0.5f;
    float fy = (((float)sy + 0.5f + dy) / 2.0f + (float)y_sampler) / h - 0.5f;
    return normalize(c.cx * fx + c.cy * fy + c.dir);
}

// sin / cos of 2*pi*u for u in (0,1) on the SFU: the argument is folded to (-pi, pi), where MUFU.SIN / MUFU.COS are
// good to ~4e-7 absolute (sin(2 pi u) = -sin(2 pi u - pi), same for cos)
__device__ __forceinline__ void sincos_2pi(float u, float& s, float& c) {
    const float x = fmaf(u, 2.0f * PI_F, -PI_F);
    s = -__sinf(x);
    c = -__cosf(x);
}

// ---- create_local_coord (src/scene.rs:112-123) ------------------------------------------------
__device__ __forceinline__ void local_coord(float3 n, float3& u, float3& v) {
    float3 a = fabsf(n.x) > 0.1f ? f3(0.f, 1.f, 0.f) : f3(1.f, 0.f, 0.f);
    u = normalize(cross(a, n));
    v = cross(n, u);
}

// ---- BRDF::eval (src/scene.rs:31-54) ---------------------------------------------------------
__device__ __forceinline__ float powi_f(float c, int p) {
    float r = 1.0f;
    for (int k = 0; k < p; ++k) r *= c;
    return r;
}
template <bool FAST = false>
__device__ __forceinline__ float3 brdf_eval(const DevMaterial& m, float3 n, float3 o, float3 i) {
    if (FAST || m.brdf == 0) return f3(m.k) * INV_PI_F;   // FAST callers only evaluate diffuse surfaces
    if (m.brdf == 1) {
        float3 r = flip_across(o, n);
        bool eq = fabsf(i.x - r.x) < 0.001f && fabsf(i.y - r.y) < 0.001f && fabsf(i.z - r.z) < 0.001f;
        if (!eq) return f3(0.f, 0.f, 0.f);
        float inv = 1.0f / dot(n, i);
        return f3(m.k) * inv;
    }
    float3 refl = flip_across(i, n);
    float c = fmaxf(dot(o, refl), 0.0f);
    int power = (int)m.k.z;
    float spec = m.k.y * (float)(power + 2) / (2.0f * PI_F) * powi_f(c, power);
    return f3(m.color_d) * (m.k.x * INV_PI_F) + f3(m.color_s) * spec;
}

// ---- BRDF::sample_incoming (src/scene.rs:56-98); xi = {u1, u2, lobe} ---------------------------
template <bool FAST = false>
__device__ __forceinline__ void brdf_sample(const DevMaterial& m, float3 n, float3 o, float4 xi, float3& i, float& pdf) {
    if (FAST || m.brdf == 0) {   // FAST callers only sample diffuse surfaces
        float z = fast_sqrt(xi.x);
        float r = fast_sqrt(1.0f - xi.x);   // sqrt(1 - z*z)
        float s, c;
        sincos_2pi(xi.y, s, c);
        float3 u, v;
        local_coord(n, u, v);
        i = normalize(u * (r * c) + v * (r * s) + n * z);
        pdf = dot(n, i) * INV_PI_F;
        return;
    }
    if (m.brdf == 1) {
        i = flip_across(o, n);
        pdf = 1.0f;
        return;
    }
    float kd = m.k.x, ks = m.k.y, p = m.k.z;
    float s, c;
    sincospif(2.0f * xi.y, &s, &c);
    if (xi.z < kd) {  // local coordinates, never rotated into the n frame (reference quirk, kept)
        float r = sqrtf(1.0f - xi.x);
        i = f3(r * c, r * s, sqrtf(xi.x));
        pdf = dot(n, i) * INV_PI_F;
    } else if (xi.z < kd + ks) {
        float r = sqrtf(1.0f - powf(xi.x, 2.0f / (p + 1.0f)));
        i = f3(r * c, r * s, powf(xi.x, 1.0f / (p + 1.0f)));
        pdf = (p + 1.0f) / (2.0f * PI_F) * powi_f(i.z, (int)p);
    } else {
        i = f3(0.f, 0.f, 0.f);
        pdf = 1.0f;
    }
}

// sphere light with its constants in the kernel parameters (the FAST instantiations): same arithmetic as the sphere
// branch of light_sample below
__device__ __forceinline__ void light_sample_sphere(const float4 L, float pdf_const, float4 xi, float3& y, float3& ny, float& pdf) {
    float z = 2.0f * xi.x - 1.0f;
    float r = fast_sqrt(fmaxf(1.0f - z * z, 0.0f));
    float s, c;
    sincos_2pi(xi.y, s, c);
    float3 n = normalize(f3(r * c, r * s, z));
    y = f3(L) + n * L.w;
    ny = n;
    pdf = pdf_const;
}

// ---- Geometry::sample for the light (src/geometry.rs:573-595); xi = {u1, u2, -, select} --------
template <bool FAST = false>
__device__ __forceinline__ void light_sample(const DevScene& S, const DevPrim* prims, const DevSceneHeader* hdr, float4 xi,
                                             float3& y, float3& ny, float& pdf) {
    if (FAST || hdr->light_geom == 0) {  // sphere: uniform over the whole surface
        const DevPrim& L = prims[hdr->light_prim];
        float z = 2.0f * xi.x - 1.0f;
        float r = fast_sqrt(fmaxf(1.0f - z * z, 0.0f));
        float s, c;
        sincos_2pi(xi.y, s, c);
        float3 n = normalize(f3(r * c, r * s, z));
        float rad = L.a.w;
        y = f3(L.a) + n * rad;
        ny = n;
        pdf = fast_rcp(4.0f * PI_F * rad * rad);
        return;
    }
    // mesh: triangle by area (WeightedIndex: partition_point(w <= chosen)), then Triangle::sample.
    // get_barycentric returns norm(b-a)*b0 + norm(c-a)*b1 WITHOUT adding `a` (src/geometry.rs:622-628).
    int n = hdr->light_n_tri;
    float chosen = xi.w * hdr->light_area;
    int lo = 0, hi = n;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (S.light_cdf[mid] <= chosen) lo = mid + 1; else hi = mid;
    }
    if (lo >= n) lo = n - 1;
    const float4* tp = S.tri_orig + (size_t)(hdr->light_first_tri + lo) * 3;
    float3 a = f3(__ldg(tp)), b = f3(__ldg(tp + 1)), c = f3(__ldg(tp + 2));
    float b0 = 1.0f - sqrtf(xi.x);
    float b1 = (1.0f - b0) * xi.y;
    y = normalize(b - a) * b0 + normalize(c - a) * b1;
    ny = normalize(cross(c - a, b - a));
    pdf = 1.0f / hdr->light_area;
}

}  // namespace rtb
