// intersect.cuh — Scene::trace_ray on the device: analytic primitives + LBVH traversal.
//
// What it must reproduce (reference, f64):
//   Scene::trace_ray            src/scene.rs:272-289   nearest hit, strict '<' (lowest index wins ties)
//   Geometry::intersect Sphere  src/geometry.rs:514-550  t > 1e-4, near root then far root, no offset
//   Geometry::intersect Plane   src/geometry.rs:551-568  |d.n| < 1e-4 miss, t >= 0, pos += 1e-5 n_facing
//   Triangle::intersect         src/geometry.rs:637-670  |n^.d| < 1e-4 miss, u,v range, t > 1e-4, +1e-5 n_facing
//   Mesh::intersect             src/geometry.rs:887-903  (brute-force branch = true nearest hit; the LBVH is
//                                                        an exact accelerator for that branch)
//   mutually_visible            src/scene.rs:258-270     visible iff nearest t + 1e-3 >= |y - x|
//
// fp32 robustness: the reference leaves a surface through a 1e-5 offset that f64 resolves and
// fp32 (ulp 7.6e-6 at x = 100) does not.  A ray therefore carries the primitive it starts on
// (`origin`), and for exactly that primitive the intersection is evaluated as the reference's
// f64 arithmetic would see it: origin 1e-5 above the facing side of a plane/triangle
// (t = -1e-5 / (d . n_facing)), or exactly on a sphere (roots 0 and 2b).  Coincident planes
// (every reference scene duplicates one wall, scenes/*.toml objects 1 and 5) share a class.
#pragma once

#include "device_types.cuh"

namespace rtb {

constexpr int STACK_SMEM = 24;   // stack levels kept in shared memory (per thread); an inner node pushes at most one
constexpr int STACK_LOCAL = 72;  // overflow levels in local memory.  The loader measures the depth of the tree it built and
                                 // refuses (RTB_EUNSUPPORTED) what does not fit BVH_MAX_DEPTH = STACK_SMEM + STACK_LOCAL levels
                                 // (lbvh.hpp; PLOC trees have no a-priori depth bound, a too deep one is rebuilt as a Karras
                                 // tree first); the spill path below additionally never writes past the array
constexpr int NODE_SENTINEL = (int)0x80000000;  // negative like a leaf, but no leaf encodes to it (first < 2^28)
constexpr float T_EPS = 1e-4f;          // sphere / triangle t threshold
constexpr float DN_EPS = 1e-4f;         // plane / triangle parallel threshold
constexpr float SURF_OFFSET = 1e-5f;    // hit-position offset along the facing normal
constexpr float SHADOW_MARGIN = 1e-3f;  // ERR_MARGIN, src/scene.rs:259

struct SharedScene {     // staged per CTA
    const DevPrim* prims;
    const DevMaterial* mats;
    int* stack;          // [STACK_SMEM][blockDim.x]
};

// dynamic shared memory needed by a CTA of `threads` threads
__host__ __device__ inline size_t shared_tables_bytes(int n_prims, int n_objects) {
    return (size_t)n_prims * sizeof(DevPrim) + (size_t)n_objects * sizeof(DevMaterial);
}
__host__ __device__ inline size_t shared_stack_bytes(int threads) { return (size_t)STACK_SMEM * threads * sizeof(int); }
__host__ __device__ inline size_t shared_scene_bytes(int n_prims, int n_objects, int threads) {
    return shared_tables_bytes(n_prims, n_objects) + shared_stack_bytes(threads);
}

// copies the primitive / material tables into shared memory (broadcast reads in the inner loops);
// with_stack: also carve the traversal stack out of the same allocation
__device__ __forceinline__ SharedScene stage_scene(const DevScene& S, unsigned char* smem, bool with_stack = true) {
    SharedScene sh;
    DevPrim* p = reinterpret_cast<DevPrim*>(smem);
    DevMaterial* m = reinterpret_cast<DevMaterial*>(smem + (size_t)S.n_prims * sizeof(DevPrim));
    int* st = reinterpret_cast<int*>(smem + shared_tables_bytes(S.n_prims, S.n_objects));
    {   // 16-byte copies; both structs are multiples of 16 B
        const float4* src = reinterpret_cast<const float4*>(S.prims);
        float4* dst = reinterpret_cast<float4*>(p);
        for (int i = threadIdx.x; i < S.n_prims * 3; i += blockDim.x) dst[i] = src[i];
        src = reinterpret_cast<const float4*>(S.mats);
        dst = reinterpret_cast<float4*>(m);
        for (int i = threadIdx.x; i < S.n_objects * 5; i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    sh.prims = p;
    sh.mats = m;
    sh.stack = with_stack ? st : nullptr;
    return sh;
}

// does the ray touch the box of all mesh triangles before tmax?  (queue class: rays that need the
// BVH vs rays whose analytic result is already final)
__device__ __forceinline__ bool ray_hits_bvh_box(const DevScene& S, float3 o, float3 d, float tmax = INFINITY) {
    if (S.n_tris == 0) return false;
    // MUFU.RCP reciprocals (2 ulp): this test only decides which queue a ray goes to, and it is widened below
    float ix = __fdividef(1.0f, fabsf(d.x) > 1e-20f ? d.x : copysignf(1e-20f, d.x));
    float iy = __fdividef(1.0f, fabsf(d.y) > 1e-20f ? d.y : copysignf(1e-20f, d.y));
    float iz = __fdividef(1.0f, fabsf(d.z) > 1e-20f ? d.z : copysignf(1e-20f, d.z));
    float x0 = (S.bvh_min.x - o.x) * ix, x1 = (S.bvh_max.x - o.x) * ix;
    float y0 = (S.bvh_min.y - o.y) * iy, y1 = (S.bvh_max.y - o.y) * iy;
    float z0 = (S.bvh_min.z - o.z) * iz, z1 = (S.bvh_max.z - o.z) * iz;
    float tmin = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), 0.0f));
    float tfar = fminf(fminf(fmaxf(x0, x1), fmaxf(y0, y1)), fminf(fmaxf(z0, z1), tmax));
    return tmin <= tfar * 1.000002f + 1e-6f;
}

// the same test for TWO rays leaving one point (extension ray | shadow ray of a vertex): the box-minus-origin terms are
// shared, the slab products are packed FP32x2, and the two chains interleave instead of sitting in separate branches
__device__ __forceinline__ void ray_pair_hits_bvh_box(const DevScene& S, float3 o, float3 d1, float tmax1, float3 d2, float tmax2,
                                                      bool& hit1, bool& hit2) {
    hit1 = hit2 = false;
    if (S.n_tris == 0) return;
    auto inv = [](float d) { return fast_rcp(fabsf(d) > 1e-20f ? d : copysignf(1e-20f, d)); };
    const float2 ix = f2(inv(d1.x), inv(d2.x)), iy = f2(inv(d1.y), inv(d2.y)), iz = f2(inv(d1.z), inv(d2.z));
    const float2 x0 = __fmul2_rn(bc(S.bvh_min.x - o.x), ix), x1 = __fmul2_rn(bc(S.bvh_max.x - o.x), ix);
    const float2 y0 = __fmul2_rn(bc(S.bvh_min.y - o.y), iy), y1 = __fmul2_rn(bc(S.bvh_max.y - o.y), iy);
    const float2 z0 = __fmul2_rn(bc(S.bvh_min.z - o.z), iz), z1 = __fmul2_rn(bc(S.bvh_max.z - o.z), iz);
    const float tmin1 = fmaxf(fmaxf(fminf(x0.x, x1.x), fminf(y0.x, y1.x)), fmaxf(fminf(z0.x, z1.x), 0.0f));
    const float tfar1 = fminf(fminf(fmaxf(x0.x, x1.x), fmaxf(y0.x, y1.x)), fminf(fmaxf(z0.x, z1.x), tmax1));
    const float tmin2 = fmaxf(fmaxf(fminf(x0.y, x1.y), fminf(y0.y, y1.y)), fmaxf(fminf(z0.y, z1.y), 0.0f));
    const float tfar2 = fminf(fminf(fmaxf(x0.y, x1.y), fmaxf(y0.y, y1.y)), fminf(fmaxf(z0.y, z1.y), tmax2));
    hit1 = tmin1 <= tfar1 * 1.000002f + 1e-6f;
    hit2 = tmin2 <= tfar2 * 1.000002f + 1e-6f;
}

// ---- analytic primitives -------------------------------------------------------------------
// prims[0, n_planes) are planes, the rest spheres; every lane walks the same table (no divergence) and the
// tests are written as selects.  `origin` = pcode of the primitive the ray starts on (PC_NONE id for camera /
// free rays): that primitive is evaluated as the reference's f64 arithmetic sees it (see the header).
// Divisions use MUFU.RCP (2 ulp) — far inside the 1e-4 relative gate on hit distances.
__device__ __forceinline__ int origin_group_of(const SharedScene& sh, uint32_t origin) {
    uint32_t id = origin & PC_ID_MASK;
    return id < TRI_BASE ? sh.prims[id].group : -1;
}

// plane k: distance along d (or a negative number / NaN-free "no hit" encoded by ok = false)
__device__ __forceinline__ float plane_t(const float4 a, float num, float3 d, bool& ok) {
    const float dn = d.x * a.x + d.y * a.y + d.z * a.z;
    const float t = num * fast_rcp(dn);
    ok = fabsf(dn) >= DN_EPS && t >= 0.0f;      // |d.n| < 1e-4 -> miss; t >= 0 (no epsilon), src/geometry.rs:551-568
    return t;
}
// numerator (pos - o).n of the plane test; for the plane class the ray starts on, the reference's origin sits
// exactly 1e-5 above the facing side, i.e. (pos - o).n_facing = -1e-5
__device__ __forceinline__ float plane_num(const DevPrim& P, float3 o, int og, uint32_t origin) {
    const float num = P.a.w - (o.x * P.a.x + o.y * P.a.y + o.z * P.a.z);
    const float self = (origin & PC_FLIPPED) ? SURF_OFFSET : -SURF_OFFSET;
    return P.group == og ? self : num;
}
// sphere: near root if > 1e-4, else far root if > 1e-4 (src/geometry.rs:514-550); origin ON the sphere: roots 0, 2b.
// det = b^2 - op.op + r^2 is evaluated as r^2 - |op - b d|^2 (same value for unit d, well conditioned in fp32).
__device__ __forceinline__ float sphere_t(float3 op, float r2, float3 d, bool self, bool& ok) {
    const float b = op.x * d.x + op.y * d.y + op.z * d.z;
    const float lx = op.x - b * d.x, ly = op.y - b * d.y, lz = op.z - b * d.z;
    const float det = r2 - (lx * lx + ly * ly + lz * lz);
    const float s = det > 0.0f ? det * rsqrtf(det) : 0.0f;
    const float tn = b - s, tf = b + s;
    float t = tn > T_EPS ? tn : tf;
    ok = det >= 0.0f && t > T_EPS;
    if (self) {
        t = 2.0f * b;
        ok = t > T_EPS;
    }
    return t;
}

// analytic half of Scene::trace_ray: nearest plane / sphere along d (strict '<': lowest index wins ties)
__device__ __forceinline__ void analytic_closest(const SharedScene& sh, int n_planes, int n_prims, float3 o, float3 d,
                                                 uint32_t origin, float& best_t, uint32_t& best_id) {
    best_t = INFINITY;
    best_id = PC_NONE;
    const int og = origin_group_of(sh, origin);
    const uint32_t oid = origin & PC_ID_MASK;
    for (int k = 0; k < n_planes; ++k) {
        const DevPrim& P = sh.prims[k];
        bool ok;
        const float t = plane_t(P.a, plane_num(P, o, og, origin), d, ok);
        if (ok && t < best_t) { best_t = t; best_id = (uint32_t)k; }
    }
    for (int k = n_planes; k < n_prims; ++k) {
        const DevPrim& P = sh.prims[k];
        bool ok;
        const float t = sphere_t(f3(P.a) - o, P.b.x, d, (uint32_t)k == oid, ok);
        if (ok && t < best_t) { best_t = t; best_id = (uint32_t)k; }
    }
}

// packed forms of plane_t / sphere_t for TWO directions (d1 | d2) = (dx, dy, dz): the same operations in the same order
// per component (FFMA2 rounds each half like fmaf), so a ray gets the same t as from the scalar functions
__device__ __forceinline__ float2 plane_t2(const float4 a, float num, float2 dx, float2 dy, float2 dz, bool& ok1, bool& ok2) {
    float2 dn = __fmul2_rn(dx, bc(a.x));
    dn = __ffma2_rn(dy, bc(a.y), dn);
    dn = __ffma2_rn(dz, bc(a.z), dn);
    const float2 t = __fmul2_rn(bc(num), f2(fast_rcp(dn.x), fast_rcp(dn.y)));
    ok1 = fabsf(dn.x) >= DN_EPS && t.x >= 0.0f;
    ok2 = fabsf(dn.y) >= DN_EPS && t.y >= 0.0f;
    return t;
}
__device__ __forceinline__ float2 sphere_t2(float3 op, float r2, float2 dx, float2 dy, float2 dz, bool self, bool& ok1, bool& ok2) {
    float2 b = __fmul2_rn(bc(op.x), dx);
    b = __ffma2_rn(bc(op.y), dy, b);
    b = __ffma2_rn(bc(op.z), dz, b);
    const float2 nb = __fmul2_rn(b, bc(-1.0f));
    const float2 lx = __ffma2_rn(nb, dx, bc(op.x)), ly = __ffma2_rn(nb, dy, bc(op.y)), lz = __ffma2_rn(nb, dz, bc(op.z));
    float2 m = __fmul2_rn(lx, lx);
    m = __ffma2_rn(ly, ly, m);
    m = __ffma2_rn(lz, lz, m);
    const float2 det = __ffma2_rn(m, bc(-1.0f), bc(r2));
    float2 s = __fmul2_rn(det, f2(rsqrtf(det.x), rsqrtf(det.y)));
    s.x = det.x > 0.0f ? s.x : 0.0f;
    s.y = det.y > 0.0f ? s.y : 0.0f;
    const float2 tn = __ffma2_rn(s, bc(-1.0f), b), tf = __fadd2_rn(b, s);
    float2 t = f2(tn.x > T_EPS ? tn.x : tf.x, tn.y > T_EPS ? tn.y : tf.y);
    ok1 = det.x >= 0.0f && t.x > T_EPS;
    ok2 = det.y >= 0.0f && t.y > T_EPS;
    if (self) {
        t = __fadd2_rn(b, b);
        ok1 = t.x > T_EPS;
        ok2 = t.y > T_EPS;
    }
    return t;
}

// Two rays leaving the same point `o` on primitive `origin` in one pass over the table:
//   d1: nearest analytic hit (t1, id1)                                  -> the extension ray
//   d2: is anything analytic in front of tlim2 ?                        -> the shadow ray (mutually_visible)
// The per-primitive set-up ((pos - o).n, c - o, the self-intersection class) is shared by both, and the two rays'
// arithmetic is issued as packed FP32x2 instructions.
__device__ __forceinline__ void analytic_pair(const SharedScene& sh, int n_planes, int n_prims, float3 o, uint32_t origin,
                                              float3 d1, float& t1, uint32_t& id1, float3 d2, float tlim2, bool& occ2) {
    t1 = INFINITY;
    id1 = PC_NONE;
    occ2 = false;
    const int og = origin_group_of(sh, origin);
    const uint32_t oid = origin & PC_ID_MASK;
    const float2 dx = f2(d1.x, d2.x), dy = f2(d1.y, d2.y), dz = f2(d1.z, d2.z);
    for (int k = 0; k < n_planes; ++k) {
        const DevPrim& P = sh.prims[k];
        const float num = plane_num(P, o, og, origin);
        bool ok1, ok2;
        const float2 t = plane_t2(P.a, num, dx, dy, dz, ok1, ok2);
        if (ok1 && t.x < t1) { t1 = t.x; id1 = (uint32_t)k; }
        occ2 |= ok2 && t.y < tlim2;
    }
    for (int k = n_planes; k < n_prims; ++k) {
        const DevPrim& P = sh.prims[k];
        const float3 op = f3(P.a) - o;
        const bool self = (uint32_t)k == oid;
        bool ok1, ok2;
        const float2 t = sphere_t2(op, P.b.x, dx, dy, dz, self, ok1, ok2);
        if (ok1 && t.x < t1) { t1 = t.x; id1 = (uint32_t)k; }
        occ2 |= ok2 && t.y < tlim2;
    }
}

// The analytic table of a scene with at most 8 primitives, carried in the KERNEL PARAMETERS: with the loops unrolled
// for a known (planes, spheres) count every coefficient is a constant-bank operand — no shared-memory loads, no loop
// counters, and the chains of different primitives interleave freely.
struct SmallScene {
    float4 a[8];        // plane: n.xyz, dot(pos, n)   sphere: centre.xyz, r
    float r2[8];
    int32_t group[8];
};
template <int NP, int NS>
__device__ __forceinline__ void analytic_pair_small(const SmallScene& ss, int og, float3 o, uint32_t origin, float3 d1, float& t1,
                                                    uint32_t& id1, float3 d2, float tlim2, bool& occ2) {
    t1 = INFINITY;
    id1 = PC_NONE;
    occ2 = false;
    const uint32_t oid = origin & PC_ID_MASK;
    const float2 dx = f2(d1.x, d2.x), dy = f2(d1.y, d2.y), dz = f2(d1.z, d2.z);
    const float self_num = (origin & PC_FLIPPED) ? SURF_OFFSET : -SURF_OFFSET;
#pragma unroll
    for (int k = 0; k < NP; ++k) {
        const float4 A = ss.a[k];
        const float num = ss.group[k] == og ? self_num : A.w - (o.x * A.x + o.y * A.y + o.z * A.z);   // plane_num
        bool ok1, ok2;
        const float2 t = plane_t2(A, num, dx, dy, dz, ok1, ok2);
        if (ok1 && t.x < t1) { t1 = t.x; id1 = (uint32_t)k; }
        occ2 |= ok2 && t.y < tlim2;
    }
#pragma unroll
    for (int k = NP; k < NP + NS; ++k) {
        const float4 A = ss.a[k];
        const float3 op = f3(A) - o;
        bool ok1, ok2;
        const float2 t = sphere_t2(op, ss.r2[k], dx, dy, dz, (uint32_t)k == oid, ok1, ok2);
        if (ok1 && t.x < t1) { t1 = t.x; id1 = (uint32_t)k; }
        occ2 |= ok2 && t.y < tlim2;
    }
}

// Any scene with at most 8 analytic primitives: unrolled over the 8 slots, each slot guarded by warp-uniform tests of
// the run-time counts (planes first, then spheres) — still constant-bank operands, no shared-memory loads, no loop counter.
__device__ __forceinline__ void analytic_pair_small8(const SmallScene& ss, int n_planes, int n_prims, int og, float3 o, uint32_t origin,
                                                     float3 d1, float& t1, uint32_t& id1, float3 d2, float tlim2, bool& occ2) {
    t1 = INFINITY;
    id1 = PC_NONE;
    occ2 = false;
    const uint32_t oid = origin & PC_ID_MASK;
    const float2 dx = f2(d1.x, d2.x), dy = f2(d1.y, d2.y), dz = f2(d1.z, d2.z);
    const float self_num = (origin & PC_FLIPPED) ? SURF_OFFSET : -SURF_OFFSET;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        const float4 A = ss.a[k];
        bool ok1 = false, ok2 = false;
        float2 t = f2(0.f, 0.f);
        if (k < n_planes) {
            const float num = ss.group[k] == og ? self_num : A.w - (o.x * A.x + o.y * A.y + o.z * A.z);
            t = plane_t2(A, num, dx, dy, dz, ok1, ok2);
        } else if (k < n_prims) {
            t = sphere_t2(f3(A) - o, ss.r2[k], dx, dy, dz, (uint32_t)k == oid, ok1, ok2);
        }
        if (ok1 && t.x < t1) { t1 = t.x; id1 = (uint32_t)k; }
        occ2 |= ok2 && t.y < tlim2;
    }
}

template <int NP, int NS>
__device__ __forceinline__ void analytic_closest_small(const SmallScene& ss, int og, float3 o, float3 d, uint32_t origin, float& best_t,
                                                       uint32_t& best_id) {
    best_t = INFINITY;
    best_id = PC_NONE;
    const uint32_t oid = origin & PC_ID_MASK;
    const float self_num = (origin & PC_FLIPPED) ? SURF_OFFSET : -SURF_OFFSET;
#pragma unroll
    for (int k = 0; k < NP; ++k) {
        const float4 A = ss.a[k];
        const float num = ss.group[k] == og ? self_num : A.w - (o.x * A.x + o.y * A.y + o.z * A.z);
        bool ok;
        const float t = plane_t(A, num, d, ok);
        if (ok && t < best_t) { best_t = t; best_id = (uint32_t)k; }
    }
#pragma unroll
    for (int k = NP; k < NP + NS; ++k) {
        const float4 A = ss.a[k];
        bool ok;
        const float t = sphere_t(f3(A) - o, ss.r2[k], d, (uint32_t)k == oid, ok);
        if (ok && t < best_t) { best_t = t; best_id = (uint32_t)k; }
    }
}

// ---- LBVH traversal ------------------------------------------------------------------------
// Per-lane traversal state.  The stack lives in shared memory (first STACK_SMEM levels, one column per
// thread) and spills to a local array beyond that.
struct Trav {
    float3 o, d;
    // slab distance of the quantised plane k of axis x: fma(8388608 + k, sx, bx) = (qmin.x + k * qstep.x - o.x) / d.x
    float sx, sy, sz, bx, by, bz;
    // PRMT selectors picking the NEAR / FAR plane of an axis out of a (lo | hi << 16) word: lo is nearer iff d > 0
    uint32_t nsx, nsy, nsz, fsx, fsy, fsz;
    uint32_t origin;     // pcode of the primitive the ray starts on
    float tlimit;        // only hits with t < tlimit count (closest: current best; any-hit: |y-x| - margin)
    uint32_t best_id;    // closest mode: id of the nearest triangle found so far (PC_NONE = none)
    int node;            // current node reference; NODE_SENTINEL = done
    int sp;
};

__device__ __forceinline__ void trav_begin(const DevScene& S, Trav& T, float3 o, float3 d, uint32_t origin, float tlimit) {
    T.o = o;
    T.d = d;
    // MUFU.RCP reciprocals (1-2 ulp).  The node boxes are quantised with QPAD = 2 grid steps of slack (lbvh.cu): the
    // constant term below carries 8388608 * s, so its rounding and the FMA's each move a plane by at most half a step.
    const float idx = __fdividef(1.0f, fabsf(d.x) > 1e-20f ? d.x : copysignf(1e-20f, d.x));
    const float idy = __fdividef(1.0f, fabsf(d.y) > 1e-20f ? d.y : copysignf(1e-20f, d.y));
    const float idz = __fdividef(1.0f, fabsf(d.z) > 1e-20f ? d.z : copysignf(1e-20f, d.z));
    T.sx = S.qstep.x * idx;
    T.sy = S.qstep.y * idy;
    T.sz = S.qstep.z * idz;
    T.bx = fmaf(-8388608.0f, T.sx, (S.qmin.x - o.x) * idx);
    T.by = fmaf(-8388608.0f, T.sy, (S.qmin.y - o.y) * idy);
    T.bz = fmaf(-8388608.0f, T.sz, (S.qmin.z - o.z) * idz);
    T.nsx = T.sx >= 0.f ? 0x7410u : 0x7432u;
    T.nsy = T.sy >= 0.f ? 0x7410u : 0x7432u;
    T.nsz = T.sz >= 0.f ? 0x7410u : 0x7432u;
    T.fsx = T.nsx ^ 0x0022u;
    T.fsy = T.nsy ^ 0x0022u;
    T.fsz = T.nsz ^ 0x0022u;
    T.origin = origin;
    T.tlimit = tlimit;
    T.best_id = PC_NONE;
    T.node = S.root;
    T.sp = 0;
}

// The shared-memory half of the stack is addressed with 32-bit shared-window addresses (ld/st.shared): `sbase` is
// the address of this thread's level-0 slot, `sstride` the byte distance between levels (blockDim.x * 4).
__device__ __forceinline__ int lds_i32(uint32_t addr) {
    int v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_i32(uint32_t addr, int v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(addr), "r"(v)); }

__device__ __forceinline__ void trav_pop(Trav& T, uint32_t sbase, uint32_t sstride, const int* lstack) {
    if (T.sp == 0) T.node = NODE_SENTINEL;
    else {
        --T.sp;
        T.node = T.sp < STACK_SMEM ? lds_i32(sbase + (uint32_t)T.sp * sstride) : lstack[T.sp - STACK_SMEM];
    }
}

// one inner node: test both child boxes, descend into the nearer hit child, push the other
template <bool COUNT>
__device__ __forceinline__ void trav_inner(const DevScene& S, Trav& T, uint32_t sbase, uint32_t sstride, int* lstack, uint32_t* work) {
    uint4 q0, q1;
    ldg256u(S.qnodes + (size_t)T.node * 2, q0, q1);
    if (COUNT) work[0]++;
    // 16-bit plane index k -> the float 8388608 + k with one PRMT (bytes k.lo, k.hi, 0x00, 0x4B), then one FMA per plane.
    // The selector already picks the plane the ray enters / leaves through (sign of d), so no per-axis min / max.
    auto pl = [](uint32_t w, uint32_t sel) { return __uint_as_float(__byte_perm(w, 0x4B000000u, sel)); };
    // packed FP32x2 FMAs (FFMA2, sm_100): x and y planes share one instruction, the z planes of the two children another —
    // 6 issue slots instead of 12 in a kernel that is bound by instruction issue
    const float2 sxy = make_float2(T.sx, T.sy), bxy = make_float2(T.bx, T.by);
    const float2 szz = make_float2(T.sz, T.sz), bzz = make_float2(T.bz, T.bz);
    const float2 n0 = __ffma2_rn(make_float2(pl(q0.x, T.nsx), pl(q0.y, T.nsy)), sxy, bxy);
    const float2 f0 = __ffma2_rn(make_float2(pl(q0.x, T.fsx), pl(q0.y, T.fsy)), sxy, bxy);
    const float2 n1 = __ffma2_rn(make_float2(pl(q0.w, T.nsx), pl(q1.x, T.nsy)), sxy, bxy);
    const float2 f1 = __ffma2_rn(make_float2(pl(q0.w, T.fsx), pl(q1.x, T.fsy)), sxy, bxy);
    const float2 nz = __ffma2_rn(make_float2(pl(q0.z, T.nsz), pl(q1.y, T.nsz)), szz, bzz);
    const float2 fz = __ffma2_rn(make_float2(pl(q0.z, T.fsz), pl(q1.y, T.fsz)), szz, bzz);
    const float n0x = n0.x, n0y = n0.y, f0x = f0.x, f0y = f0.y, n1x = n1.x, n1y = n1.y, f1x = f1.x, f1y = f1.y;
    const float n0z = nz.x, n1z = nz.y, f0z = fz.x, f1z = fz.y;
    const float tmin0 = fmaxf(fmaxf(n0x, n0y), fmaxf(n0z, 0.0f));
    const float tmax0 = fminf(fminf(f0x, f0y), fminf(f0z, T.tlimit));
    const float tmin1 = fmaxf(fmaxf(n1x, n1y), fmaxf(n1z, 0.0f));
    const float tmax1 = fminf(fminf(f1x, f1y), fminf(f1z, T.tlimit));
    const bool h0 = tmin0 <= tmax0, h1 = tmin1 <= tmax1;
    const int c0 = (int)q1.z, c1 = (int)q1.w;
    // Select-based step (no three-way branch): the lane always peeks at its stack top; "both hit" pushes the
    // farther child, "none hit" pops.  Only the (rare) spill beyond STACK_SMEM levels branches.
    const bool both = h0 && h1, none = !h0 && !h1;
    const bool swap = tmin1 < tmin0;
    const int nearc = both ? (swap ? c1 : c0) : (h0 ? c0 : c1);
    const int farc = swap ? c0 : c1;
    if (T.sp < STACK_SMEM) {
        const uint32_t slot = sbase + (uint32_t)max(T.sp - (none ? 1 : 0), 0) * sstride;   // push target, or the top entry when popping
        const int top = lds_i32(slot);
        if (both) sts_i32(slot, farc);
        T.node = none ? (T.sp == 0 ? NODE_SENTINEL : top) : nearc;
        T.sp += both ? 1 : (none && T.sp > 0 ? -1 : 0);
    } else {  // spill levels (local memory); T.sp == STACK_SMEM pops from shared memory via trav_pop
        if (both) {
            if (T.sp - STACK_SMEM < STACK_LOCAL) {   // cannot fail for a tree the loader accepted; never write past the array
                lstack[T.sp - STACK_SMEM] = farc;
                ++T.sp;
            }
            T.node = nearc;
        } else if (none) {
            trav_pop(T, sbase, sstride, lstack);
        } else {
            T.node = nearc;
        }
    }
}

// one leaf (T.node < 0, not the sentinel): Triangle::intersect on its 1..8 triangles.
// ANY_HIT: returns true at the first triangle with t < tlimit.  Closest: shrinks tlimit / records best_id.
template <bool ANY_HIT, bool COUNT>
__device__ __forceinline__ bool trav_leaf(const DevScene& S, Trav& T, uint32_t* work) {
    const uint32_t v = ~(uint32_t)T.node;
    const uint32_t first = v >> 3, cnt = (v & 7u) + 1u;
    const uint32_t origin_id = T.origin & PC_ID_MASK;
    for (uint32_t s = first; s < first + cnt; ++s) {
        const float4* tp = S.tris + (size_t)s * TRI_STRIDE;
        float4 t0, t1;
        ldg256(tp, t0, t1);
        const float4 t2 = __ldg(tp + 2);
        if (COUNT) work[1]++;
        float3 e1 = f3(t1), e2 = f3(t2);
        float3 pvec = cross(T.d, e2);
        float det = dot(e1, pvec);      // = d . ((c-a) x (b-a)) = |N| (n^ . d)
        float nd = det * t0.w;          // n^ . d
        if (fabsf(nd) < DN_EPS) continue;
        float inv = __fdividef(1.0f, det);   // 2 ulp: far inside the 1e-4 distance gate
        float3 tvec = T.o - f3(t0);
        float u = dot(tvec, pvec) * inv;
        float3 qvec = cross(tvec, e1);
        float vv = dot(T.d, qvec) * inv;
        float t = dot(e2, qvec) * inv;
        if (TRI_BASE + s == origin_id) {  // the triangle this ray starts on (see header)
            float dnf = (T.origin & PC_FLIPPED) ? -nd : nd;
            t = -SURF_OFFSET / dnf;
        }
        if (u < 0.0f || vv < 0.0f || u + vv > 1.0f || !(t > T_EPS)) continue;
        if (t < T.tlimit) {
            if (ANY_HIT) return true;
            T.tlimit = t;
            T.best_id = TRI_BASE + s;
        }
    }
    return false;
}

// whole traversal for one ray ("while-while": a lane leaves the inner-node loop when it holds a leaf,
// so the triangle code runs with as many lanes as possible)
template <bool ANY_HIT, bool COUNT>
__device__ __forceinline__ bool bvh_traverse(const DevScene& S, const SharedScene& sh, float3 o, float3 d, uint32_t origin,
                                             float& best_t, uint32_t& best_id, float dist, uint32_t* work) {
    // ANY_HIT: returns true as soon as some triangle has t + SHADOW_MARGIN < dist.
    // else   : updates (best_t, best_id) with the nearest triangle hit below best_t.
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(sh.stack + threadIdx.x), sstride = blockDim.x * 4u;
    int lstack[STACK_LOCAL];
    Trav T;
    trav_begin(S, T, o, d, origin, ANY_HIT ? dist - SHADOW_MARGIN : best_t);
    while (T.node != NODE_SENTINEL) {
        while (T.node >= 0) trav_inner<COUNT>(S, T, sbase, sstride, lstack, work);
        if (T.node != NODE_SENTINEL) {
            if (trav_leaf<ANY_HIT, COUNT>(S, T, work)) return true;
            trav_pop(T, sbase, sstride, lstack);
        }
    }
    if (!ANY_HIT && T.best_id != PC_NONE) {
        best_t = T.tlimit;
        best_id = T.best_id;
    }
    return false;
}

// ---- hit geometry ----------------------------------------------------------------------------
struct HitGeom {
    float3 pos;      // Hit.pos (offset rules of the reference applied)
    float3 n;        // Hit.n, facing the ray
    int obj;         // Hit.id
    uint32_t pcode;  // id | PC_FLIPPED
};

// tri_n: the triangle's (unit normal | object id) record, fetched early by the caller (ignored for analytic ids)
__device__ __forceinline__ HitGeom hit_geometry(const SharedScene& sh, float3 o, float3 d, float t, uint32_t id, float4 tri_n) {
    HitGeom h;
    float3 p = o + t * d;
    float3 n;
    bool offset = true;
    if (id < TRI_BASE) {
        const DevPrim& P = sh.prims[id];
        h.obj = P.obj;
        if (P.type == 0) n = f3(P.a);
        else { n = normalize(p - f3(P.a)); offset = false; }
    } else {
        n = f3(tri_n);  // Triangle::normal: norm((c-a) x (b-a))
        h.obj = __float_as_int(tri_n.w);
    }
    bool flipped = !(dot(n, -d) >= 0.0f);
    if (flipped) n = -n;
    h.n = n;
    h.pos = offset ? p + SURF_OFFSET * n : p;
    h.pcode = id | (flipped ? PC_FLIPPED : 0u);
    return h;
}

}  // namespace rtb
