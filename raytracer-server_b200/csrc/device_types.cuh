// device_types.cuh — device-side scene layout (structure of arrays, fp32) and small math helpers.
//
// Replaces the reference's AoS f64 scene graph (Object / Geometry / Mesh / Octree,
// src/scene.rs:10-28,101-107, src/geometry.rs:371-424,1133-1143):
//   * analytic primitives (planes, spheres) and per-object materials: small tables that every
//     CTA stages into shared memory once (broadcast reads in the inner loops);
//   * all mesh triangles of all objects: one LBVH (lbvh.cu), 64-byte nodes holding both child
//     boxes, triangles in leaf order as three float4 (v0|1/|N|, e1|global tri id, e2|object id).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace rtb {

// ---------------------------------------------------------------- primitive codes
// pcode: bit31 = hit normal flipped w.r.t. the geometric normal, bit30 = previous vertex was
// specular (emission + ks/p still to be applied), bit29 = `o` is stale (reference quirk,
// src/scene.rs:178), bit28 = the ray is a BRDF sample of the balance-heuristic estimator (RTB_EST_MIS_BALANCE: its pdf
// rides in the `ov` slot, the light's emission is still to be added with the MIS weight),
// bits 0..27 = id: analytic primitive index (< TRI_BASE) or TRI_BASE + leaf slot.
constexpr uint32_t PC_FLIPPED = 0x80000000u;
constexpr uint32_t PC_SPEC_PENDING = 0x40000000u;
constexpr uint32_t PC_STALE_O = 0x20000000u;
constexpr uint32_t PC_MIS_PENDING = 0x10000000u;
constexpr uint32_t PC_ID_MASK = 0x0fffffffu;
constexpr uint32_t PC_NONE = 0x0fffffffu;
constexpr uint32_t TRI_BASE = 256u;  // == MAX_OBJECTS
constexpr int TRI_STRIDE = 4;        // float4 per LBVH triangle record: 48 B of data padded to 64 B so that the first 32 B
                                     // can be fetched by one 256-bit load

struct DevPrim {      // 48 B, mirrors FlatPrim
    float4 a;         // plane: n.xyz, dot(pos,n)   sphere: c.xyz, r
    float4 b;         // plane: pos.xyz             sphere: r*r
    int32_t type, obj, group, pad;
};

struct DevMaterial {  // 80 B, mirrors FlatMaterial
    float4 emitted;
    float4 k;
    float4 color_d;
    float4 color_s;
    int32_t brdf, geom, first_tri, n_tri;
};

struct DevSceneHeader {  // lives in global memory; one per scene
    float cam_pos[3];
    float cam_dir[3];
    int32_t n_prims;
    int32_t n_objects;
    int32_t light_obj;
    int32_t light_geom;    // GEOM_*
    int32_t light_prim;    // analytic index of the light when it is a sphere
    int32_t light_first_tri, light_n_tri;
    float light_area;      // Mesh::surface_area of the UNTRANSFORMED mesh (reference quirk)
    int32_t n_tris;
    int32_t root;          // encoded BVH root reference (inner >= 0, leaf < 0), valid if n_tris > 0
    float bvh_min[3];
    float bvh_max[3];
    // the light table of RTB_EST_NEE_ALL_LIGHTS (light_rule.cuh, DESIGN §3f).  The offsets count 256-byte units from the header
    // (every staged table starts on such a boundary), so they reach past 4 GB of scene while the header keeps 4-byte fields.
    int32_t n_lights;
    int32_t lights_select;   // 1: a vertex draws block 1 for the choice (more than one light, or a mesh light)
    int32_t off_lights;      // DevLight[n_lights]
    int32_t off_light_cdf;   // float[]: the lights' cdf (n_lights entries), then one triangle cdf per mesh light
    int32_t off_light_of;    // int32_t[n_objects]: each object's table entry, -1 = not in the table
};

struct DevScene {          // passed to kernels by value
    const DevSceneHeader* hdr;
    const DevPrim* prims;
    const DevMaterial* mats;
    const uint4* qnodes;   // 2 x uint4 per node: the 16-bit quantised table the traversal reads (lbvh.cu)
    float3 qmin, qstep;    // quantisation grid of qnodes
    const float4* tris;    // TRI_STRIDE x float4 per triangle (3 used), leaf order
    const float4* tri_nrm; // unit geometric normal | object id per triangle, leaf order (shading)
    const float* light_cdf;
    const float4* tri_orig; // 3 x float4 per triangle in GLOBAL order: a, b, c (mesh-light sampling)
    // RTB_ACCEL_OCTREE_REFERENCE (octree.cuh): the reference's per-mesh octrees, built lazily on first use (nullptr before)
    const float4* oct_nodes;   // 2 x float4 per node (octree.cuh)
    const float4* oct_tris;    // leaf triangles in reference order: a COPY of the `tris` record per reference (TRI_STRIDE x float4), its slot in `tris` in [1].w
    const int32_t* oct_roots;  // root node per mesh, in object order (-1: empty mesh)
    int32_t n_oct_meshes;
    int32_t n_prims, n_objects, n_tris, root;
    int32_t n_planes;      // prims[0, n_planes) are planes, prims[n_planes, n_prims) spheres
    float3 bvh_min, bvh_max;
};

// 256-bit read-only load (LDG.E.256, sm_100+; p must be 32-byte aligned).  k_traverse is bound by the L1 data pipe,
// which spends one wavefront per 128-byte line an instruction touches — a divergent lane costs the same wavefront
// for 16 or for 32 bytes, so fetching a 64-byte node with two loads instead of four halves that cost.
__device__ __forceinline__ void ldg256u(const uint4* p, uint4& a, uint4& b) {
    asm("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w), "=r"(b.x), "=r"(b.y), "=r"(b.z), "=r"(b.w)
        : "l"(p));
}
__device__ __forceinline__ void ldg256(const float4* p, float4& a, float4& b) {
    asm("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
        : "l"(p));
}

// ---------------------------------------------------------------- float3 helpers
__host__ __device__ __forceinline__ float3 f3(float x, float y, float z) { return make_float3(x, y, z); }
__host__ __device__ __forceinline__ float3 f3(const float4& v) { return make_float3(v.x, v.y, v.z); }
__host__ __device__ __forceinline__ float3 operator+(float3 a, float3 b) { return f3(a.x + b.x, a.y + b.y, a.z + b.z); }
__host__ __device__ __forceinline__ float3 operator-(float3 a, float3 b) { return f3(a.x - b.x, a.y - b.y, a.z - b.z); }
__host__ __device__ __forceinline__ float3 operator-(float3 a) { return f3(-a.x, -a.y, -a.z); }
__host__ __device__ __forceinline__ float3 operator*(float3 a, float s) { return f3(a.x * s, a.y * s, a.z * s); }
__host__ __device__ __forceinline__ float3 operator*(float s, float3 a) { return f3(a.x * s, a.y * s, a.z * s); }
__host__ __device__ __forceinline__ float3 operator*(float3 a, float3 b) { return f3(a.x * b.x, a.y * b.y, a.z * b.z); }
__host__ __device__ __forceinline__ float dot(float3 a, float3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__host__ __device__ __forceinline__ float3 cross(float3 a, float3 b) {
    return f3(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
__device__ __forceinline__ float3 normalize(float3 a) {
    float inv = rsqrtf(dot(a, a));
    return a * inv;
}
// single-instruction SFU forms (MUFU.SQRT / MUFU.RCP, ~1 ulp, denormals flushed) for the sampling arithmetic: IEEE sqrtf /
// division are 8-10 instruction sequences with a slow-path call each
__device__ __forceinline__ float fast_sqrt(float x) { float r; asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ float fast_rcp(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
// packed FP32x2 helpers (FFMA2 / FMUL2, sm_100): the kernels are bound by instruction issue, and two rays that meet the
// same primitive do the same arithmetic — one issue slot for both.  bc() = a scalar both halves use (SASS takes it as
// a broadcast .F32 operand, no extra register)
__device__ __forceinline__ float2 f2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 bc(float a) { return make_float2(a, a); }
// per-thread asynchronous global -> shared copies (LDGSTS): the prefetched queue entry of a k_shade lane lives in
// shared memory instead of 18 registers; wait_all makes the thread's own copies visible to it
__device__ __forceinline__ void cp_async16(uint32_t saddr, const void* g) { asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(saddr), "l"(g)); }
__device__ __forceinline__ void cp_async8(uint32_t saddr, const void* g) { asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(saddr), "l"(g)); }
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ float4 lds_f4(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}
__device__ __forceinline__ float2 lds_f2(uint32_t saddr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(saddr));
    return v;
}
// atomicAdd as ONE instruction.  nvcc rewrites atomicAdd(uniform address) into a warp-aggregated sequence (VOTE / POPC /
// ATOMG by the leader / SHFL of the result), and the SHFL waits for the atomic's round trip on the spot — which defeats a
// reservation that is issued ahead precisely so that nobody waits for it.  Called by one lane; the result is read later.
__device__ __forceinline__ uint32_t atomic_add_lane(uint32_t* p, uint32_t v) {
    uint32_t old;
    asm volatile("atom.global.add.u32 %0, [%1], %2;" : "=r"(old) : "l"(p), "r"(v) : "memory");
    return old;
}
// Vec3::flip_across (src/geometry.rs:99-101)
__device__ __forceinline__ float3 flip_across(float3 s, float3 axis) { return (2.0f * dot(s, axis)) * axis - s; }

}  // namespace rtb
