// lbvh.cu — device-built linear BVH over all mesh triangles of a scene.
//
// Replaces the reference's per-mesh octree (Octree::build / _build, src/geometry.rs:1149-1216,
// set-up time only) with a structure that answers the question the reference's own brute-force
// branch answers (Mesh::intersect, src/geometry.rs:887-903): the true nearest triangle.
//
// Pipeline (all on the GPU, one stream):
//   1. triangle bounds + centroid bounds (atomic min/max on order-preserving int keys)
//   2. hierarchy, one of
//        binned SAH (default, round 2)  top-down, level-synchronous, 16 bins per axis, leaves of <= 2 triangles: see the
//               k_sah_* kernels.  Emits nodes and leaf order directly (steps 3-5 below are for the two bottom-up builders).
//        PLOC   (RTB_BVH=ploc; the default of round 1) parallel locally-ordered clustering, Meister & Bittner 2018: mutual
//               nearest neighbours (by merged box area, +-16 positions in Morton order) merge round by round;
//               depth-first leaf positions by walking parent links
//        Karras (RTB_BVH=lbvh; the fallback when a tree comes out deeper than the traversal stack) Karras 2012: one thread per
//               internal node finds its range and split, bottom-up refit with one atomic arrival counter per node
//      Measured on flying_unicorn 1920x1080x64 (k_traverse per frame, tools/gpu_bvh_quality.py): Karras 60.6 ms, PLOC 59.4 ms,
//      binned SAH 54.8 ms (the host prototype with a full sweep instead of bins: 54.3 ms).  Build: 6 ms more than PLOC.
//   3. 63-bit Morton codes of the centroids (21 bits per axis), radix sort of (code, triangle) pairs   [cub::DeviceRadixSort]
//   4. PLOC / Karras hierarchy over the sorted triangles
//   5. collapse subtrees of <= LEAF_MAX triangles into leaves (subtrees are contiguous in leaf order),
//      compact the surviving nodes                                   [cub::DeviceScan]
//   6. emit 64-byte nodes {child0 box, child1 box, child refs} and triangles in leaf order
#include "lbvh.hpp"
#include "device_types.cuh"

#include <cub/cub.cuh>

#include <algorithm>
#include <cfloat>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

namespace rtb {
namespace {

#define LBVH_CHECK(x)                                                                  \
    do {                                                                               \
        cudaError_t e_ = (x);                                                          \
        if (e_ != cudaSuccess) {                                                       \
            err = std::string("CUDA error in LBVH build: ") + cudaGetErrorString(e_); \
            return false;                                                              \
        }                                                                              \
    } while (0)

constexpr int LEAF_MAX = 2;

int depth_limit() {   // levels the traversal stack holds; RTB_BVH_MAX_DEPTH lowers it (test hook)
    int d = BVH_MAX_DEPTH;
    if (const char* e = getenv("RTB_BVH_MAX_DEPTH")) d = std::min(BVH_MAX_DEPTH, std::max(1, atoi(e)));
    return d;
}

__device__ __forceinline__ int float_to_ordered(float f) {
    int i = __float_as_int(f);
    return i >= 0 ? i : i ^ 0x7fffffff;
}
__device__ __forceinline__ float ordered_to_float(int i) { return __int_as_float(i >= 0 ? i : i ^ 0x7fffffff); }

struct Bounds6 {
    int lo[3], hi[3];    // triangle-vertex bounds (ordered ints)
    int clo[3], chi[3];  // centroid bounds
};

__global__ void k_init_bounds(Bounds6* b) {
    for (int k = 0; k < 3; ++k) {
        b->lo[k] = b->clo[k] = float_to_ordered(FLT_MAX);
        b->hi[k] = b->chi[k] = float_to_ordered(-FLT_MAX);
    }
}

__global__ void k_tri_bounds(const float* __restrict__ verts, int n, float4* __restrict__ lo4, float4* __restrict__ hi4, Bounds6* gb) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* v = verts + (size_t)i * 9;
    float lo[3], hi[3];
    for (int k = 0; k < 3; ++k) {
        float a = v[k], b = v[3 + k], c = v[6 + k];
        lo[k] = fminf(a, fminf(b, c));
        hi[k] = fmaxf(a, fmaxf(b, c));
    }
    for (int k = 0; k < 3; ++k) {  // conservative pad (the traversal uses approximate reciprocals)
        float pad = fmaxf(fabsf(lo[k]), fabsf(hi[k])) * 1e-6f + 1e-30f;
        lo[k] -= pad;
        hi[k] += pad;
    }
    lo4[i] = make_float4(lo[0], lo[1], lo[2], 0.f);
    hi4[i] = make_float4(hi[0], hi[1], hi[2], 0.f);
    for (int k = 0; k < 3; ++k) {
        float c = 0.5f * (lo[k] + hi[k]);
        atomicMin(&gb->lo[k], float_to_ordered(lo[k]));
        atomicMax(&gb->hi[k], float_to_ordered(hi[k]));
        atomicMin(&gb->clo[k], float_to_ordered(c));
        atomicMax(&gb->chi[k], float_to_ordered(c));
    }
}

__device__ __forceinline__ unsigned long long expand21(unsigned long long v) {  // 21 bits -> every third bit
    v &= 0x1fffffull;
    v = (v | v << 32) & 0x1f00000000ffffull;
    v = (v | v << 16) & 0x1f0000ff0000ffull;
    v = (v | v << 8) & 0x100f00f00f00f00full;
    v = (v | v << 4) & 0x10c30c30c30c30c3ull;
    v = (v | v << 2) & 0x1249249249249249ull;
    return v;
}

__global__ void k_morton(const float4* __restrict__ lo4, const float4* __restrict__ hi4, int n, const Bounds6* gb,
                         unsigned long long* __restrict__ keys, uint32_t* __restrict__ vals) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 lo = lo4[i], hi = hi4[i];
    float c[3] = {0.5f * (lo.x + hi.x), 0.5f * (lo.y + hi.y), 0.5f * (lo.z + hi.z)};
    unsigned long long q[3];
    for (int k = 0; k < 3; ++k) {
        float a = ordered_to_float(gb->clo[k]), b = ordered_to_float(gb->chi[k]);
        float ext = b - a;
        float u = ext > 0.f ? (c[k] - a) / ext : 0.f;
        u = fminf(fmaxf(u, 0.f), 1.f);
        q[k] = (unsigned long long)fminf(u * 2097152.0f, 2097151.0f);
    }
    keys[i] = (expand21(q[0]) << 2) | (expand21(q[1]) << 1) | expand21(q[2]);
    vals[i] = (uint32_t)i;
}

// common-prefix length of sorted keys i and j; ties are broken by the index (Karras 2012, sec. 4)
__device__ __forceinline__ int delta(const unsigned long long* keys, int n, int i, int j) {
    if (j < 0 || j >= n) return -1;
    unsigned long long a = keys[i], b = keys[j];
    if (a == b) return 64 + __clz(i ^ j);
    return __clzll(a ^ b);
}

// child reference during the build: >= 0 internal node, < 0 leaf slot ~ref
__global__ void k_hierarchy(const unsigned long long* __restrict__ keys, int n, int* __restrict__ left, int* __restrict__ right,
                            int* __restrict__ parent_int, int* __restrict__ parent_leaf, int* __restrict__ rfirst,
                            int* __restrict__ rlast) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n - 1) return;
    int d = delta(keys, n, i, i + 1) - delta(keys, n, i, i - 1) >= 0 ? 1 : -1;
    int dmin = delta(keys, n, i, i - d);
    int lmax = 2;
    while (delta(keys, n, i, i + lmax * d) > dmin) lmax *= 2;
    int l = 0;
    for (int t = lmax / 2; t >= 1; t /= 2)
        if (delta(keys, n, i, i + (l + t) * d) > dmin) l += t;
    int j = i + l * d;
    int dnode = delta(keys, n, i, j);
    int s = 0;
    for (int t = (l + 1) / 2;; t = (t + 1) / 2) {
        if (delta(keys, n, i, i + (s + t) * d) > dnode) s += t;
        if (t == 1) break;
    }
    int gamma = i + s * d + min(d, 0);
    int first = min(i, j), last = max(i, j);
    int lc = (first == gamma) ? ~gamma : gamma;
    int rc = (last == gamma + 1) ? ~(gamma + 1) : gamma + 1;
    left[i] = lc;
    right[i] = rc;
    rfirst[i] = first;
    rlast[i] = last;
    if (lc >= 0) parent_int[lc] = i; else parent_leaf[~lc] = i;
    if (rc >= 0) parent_int[rc] = i; else parent_leaf[~rc] = i;
    if (i == 0) parent_int[0] = -1;
}

__global__ void k_refit(int n, const uint32_t* __restrict__ sorted, const float4* __restrict__ tlo, const float4* __restrict__ thi,
                        const int* __restrict__ left, const int* __restrict__ right, const int* __restrict__ parent_int,
                        const int* __restrict__ parent_leaf, int* __restrict__ arrive, float4* __restrict__ nlo,
                        float4* __restrict__ nhi) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    int node = parent_leaf[s];
    while (node >= 0) {
        if (atomicAdd(&arrive[node], 1) == 0) return;  // first child to arrive leaves; the second one merges
        __threadfence();
        int lc = left[node], rc = right[node];
        float4 alo = lc >= 0 ? __ldcg(&nlo[lc]) : tlo[sorted[~lc]], ahi = lc >= 0 ? __ldcg(&nhi[lc]) : thi[sorted[~lc]];
        float4 blo = rc >= 0 ? __ldcg(&nlo[rc]) : tlo[sorted[~rc]], bhi = rc >= 0 ? __ldcg(&nhi[rc]) : thi[sorted[~rc]];
        nlo[node] = make_float4(fminf(alo.x, blo.x), fminf(alo.y, blo.y), fminf(alo.z, blo.z), 0.f);
        nhi[node] = make_float4(fmaxf(ahi.x, bhi.x), fmaxf(ahi.y, bhi.y), fmaxf(ahi.z, bhi.z), 0.f);
        __threadfence();
        node = parent_int[node];
    }
}

__global__ void k_mark_used(int n_internal, int leaf_max, const int* __restrict__ rfirst, const int* __restrict__ rlast, int* __restrict__ used) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_internal) return;
    used[i] = (rlast[i] - rfirst[i] + 1) > leaf_max ? 1 : 0;
}

__device__ __forceinline__ int encode_leaf(int first, int count) { return ~((first << 3) | (count - 1)); }

__global__ void k_emit(int n_internal, const uint32_t* __restrict__ sorted, const float4* __restrict__ tlo,
                       const float4* __restrict__ thi, const int* __restrict__ left, const int* __restrict__ right,
                       const int* __restrict__ rfirst, const int* __restrict__ rlast, const int* __restrict__ used,
                       const int* __restrict__ newidx, const float4* __restrict__ nlo, const float4* __restrict__ nhi,
                       float4* __restrict__ out, const int* __restrict__ leafpos) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_internal || !used[i]) return;
    int c[2] = {left[i], right[i]};
    float4 lo[2], hi[2];
    int ref[2];
    for (int k = 0; k < 2; ++k) {
        if (c[k] < 0) {
            int s = ~c[k];
            lo[k] = tlo[sorted[s]];
            hi[k] = thi[sorted[s]];
            ref[k] = encode_leaf(leafpos ? leafpos[s] : s, 1);
        } else {
            lo[k] = nlo[c[k]];
            hi[k] = nhi[c[k]];
            ref[k] = used[c[k]] ? newidx[c[k]] : encode_leaf(rfirst[c[k]], rlast[c[k]] - rfirst[c[k]] + 1);
        }
    }
    float4* o = out + (size_t)newidx[i] * 4;
    o[0] = make_float4(lo[0].x, hi[0].x, lo[0].y, hi[0].y);
    o[1] = make_float4(lo[1].x, hi[1].x, lo[1].y, hi[1].y);
    o[2] = make_float4(lo[0].z, hi[0].z, lo[1].z, hi[1].z);
    o[3] = make_float4(__int_as_float(ref[0]), __int_as_float(ref[1]), 0.f, 0.f);
}

__global__ void k_pack_tris(int n, const uint32_t* __restrict__ sorted, const float* __restrict__ verts,
                            const int32_t* __restrict__ tri_obj, float4* __restrict__ out, float4* __restrict__ nrm) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    uint32_t g = sorted[s];
    const float* v = verts + (size_t)g * 9;
    float3 a = make_float3(v[0], v[1], v[2]);
    float3 e1 = make_float3(v[3] - a.x, v[4] - a.y, v[5] - a.z);  // b - a
    float3 e2 = make_float3(v[6] - a.x, v[7] - a.y, v[8] - a.z);  // c - a
    // N = (c-a) x (b-a)  (Triangle::normal, src/geometry.rs:606-608)
    float nx = e2.y * e1.z - e2.z * e1.y, ny = e2.z * e1.x - e2.x * e1.z, nz = e2.x * e1.y - e2.y * e1.x;
    float len = sqrtf(nx * nx + ny * ny + nz * nz);
    float4* o = out + (size_t)s * rtb::TRI_STRIDE;
    o[3] = make_float4(0.f, 0.f, 0.f, 0.f);
    o[0] = make_float4(a.x, a.y, a.z, len > 0.f ? 1.0f / len : 0.f);
    o[1] = make_float4(e1.x, e1.y, e1.z, __int_as_float((int)g));
    o[2] = make_float4(e2.x, e2.y, e2.z, __int_as_float(tri_obj[g]));
    float il = len > 0.f ? 1.0f / len : 0.f;
    nrm[s] = make_float4(nx * il, ny * il, nz * il, __int_as_float(tri_obj[g]));
}

// ---------------------------------------------------------------- PLOC (parallel locally-ordered clustering)
// Meister & Bittner 2018: the Morton-sorted triangles are clusters; every round each cluster looks PLOC_RADIUS
// neighbours to either side for the partner that gives the smallest merged box area, mutual nearest neighbours
// merge.  Same inputs as the Karras hierarchy above, markedly better trees (bottom-up, surface-area driven).
constexpr int PLOC_RADIUS = 16;

__device__ __forceinline__ float box_area(float4 lo, float4 hi) {
    float dx = hi.x - lo.x, dy = hi.y - lo.y, dz = hi.z - lo.z;
    return dx * dy + dy * dz + dz * dx;
}

__global__ void k_ploc_init(int n, const uint32_t* __restrict__ sorted, const float4* __restrict__ tlo, const float4* __restrict__ thi,
                            int* __restrict__ cnode, float4* __restrict__ clo, float4* __restrict__ chi, int* __restrict__ csize) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    cnode[s] = ~s;
    clo[s] = tlo[sorted[s]];
    chi[s] = thi[sorted[s]];
    csize[s] = 1;
}

__global__ void k_ploc_nn(int m, int radius, const float4* __restrict__ clo, const float4* __restrict__ chi, int* __restrict__ nn) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const float4 lo = clo[i], hi = chi[i];
    float best = FLT_MAX;
    int bj = -1;
    const int j0 = max(0, i - radius), j1 = min(m - 1, i + radius);
    for (int j = j0; j <= j1; ++j) {
        if (j == i) continue;
        const float4 l2 = clo[j], h2 = chi[j];
        float4 ul = make_float4(fminf(lo.x, l2.x), fminf(lo.y, l2.y), fminf(lo.z, l2.z), 0.f);
        float4 uh = make_float4(fmaxf(hi.x, h2.x), fmaxf(hi.y, h2.y), fmaxf(hi.z, h2.z), 0.f);
        float a = box_area(ul, uh);
        if (a < best) { best = a; bj = j; }   // ties: the lower index, on both sides -> mutual pairs exist
    }
    nn[i] = bj;
}

__global__ void k_ploc_flags(int m, const int* __restrict__ nn, int* __restrict__ valid, int* __restrict__ merge) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m) return;
    const int j = nn[i];
    const bool mutual = j >= 0 && nn[j] == i;
    valid[i] = (mutual && j < i) ? 0 : 1;   // the higher-indexed partner disappears
    merge[i] = (mutual && i < j) ? 1 : 0;   // the lower-indexed partner becomes the merged cluster
}

__global__ void k_ploc_apply(int m, const int* __restrict__ cnode, const float4* __restrict__ clo, const float4* __restrict__ chi,
                             const int* __restrict__ csize, const int* __restrict__ nn, const int* __restrict__ valid,
                             const int* __restrict__ merge, const int* __restrict__ pv, const int* __restrict__ pm, int node_base,
                             int* __restrict__ ocnode, float4* __restrict__ oclo, float4* __restrict__ ochi, int* __restrict__ ocsize,
                             int* __restrict__ left, int* __restrict__ right, float4* __restrict__ nlo, float4* __restrict__ nhi,
                             int* __restrict__ nsize, int* __restrict__ parent_int, int* __restrict__ parent_leaf,
                             unsigned char* __restrict__ isright_int, unsigned char* __restrict__ isright_leaf) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= m || !valid[i]) return;
    const int p = pv[i];
    if (!merge[i]) {
        ocnode[p] = cnode[i];
        oclo[p] = clo[i];
        ochi[p] = chi[i];
        ocsize[p] = csize[i];
        return;
    }
    const int j = nn[i];
    const int idx = node_base + pm[i];
    const int a = cnode[i], b = cnode[j];
    const float4 l1 = clo[i], h1 = chi[i], l2 = clo[j], h2 = chi[j];
    const float4 ul = make_float4(fminf(l1.x, l2.x), fminf(l1.y, l2.y), fminf(l1.z, l2.z), 0.f);
    const float4 uh = make_float4(fmaxf(h1.x, h2.x), fmaxf(h1.y, h2.y), fmaxf(h1.z, h2.z), 0.f);
    left[idx] = a;
    right[idx] = b;
    nlo[idx] = ul;
    nhi[idx] = uh;
    nsize[idx] = csize[i] + csize[j];
    if (a >= 0) { parent_int[a] = idx; isright_int[a] = 0; } else { parent_leaf[~a] = idx; isright_leaf[~a] = 0; }
    if (b >= 0) { parent_int[b] = idx; isright_int[b] = 1; } else { parent_leaf[~b] = idx; isright_leaf[~b] = 1; }
    ocnode[p] = idx;
    oclo[p] = ul;
    ochi[p] = uh;
    ocsize[p] = csize[i] + csize[j];
}

// position of every leaf / first leaf of every internal node in depth-first (left before right) order:
// walking up, every time we come out of a right child the whole left sibling lies before us
__global__ void k_ploc_positions(int n, int n_internal, const int* __restrict__ left, const int* __restrict__ nsize,
                                 const int* __restrict__ parent_int, const int* __restrict__ parent_leaf,
                                 const unsigned char* __restrict__ isright_int, const unsigned char* __restrict__ isright_leaf,
                                 int* __restrict__ leafpos, int* __restrict__ rfirst, int* __restrict__ rlast) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n + n_internal) return;
    const bool is_leaf = t < n;
    const int me = is_leaf ? t : t - n;
    int p = is_leaf ? parent_leaf[me] : parent_int[me];
    bool r = is_leaf ? isright_leaf[me] != 0 : isright_int[me] != 0;
    int pos = 0;
    while (p >= 0) {
        if (r) { const int l = left[p]; pos += l >= 0 ? nsize[l] : 1; }
        r = isright_int[p] != 0;
        p = parent_int[p];
    }
    if (is_leaf) leafpos[me] = pos;
    else { rfirst[me] = pos; rlast[me] = pos + nsize[me] - 1; }
}

__global__ void k_ploc_order(int n, const uint32_t* __restrict__ sorted, const int* __restrict__ leafpos, uint32_t* __restrict__ order) {
    int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s < n) order[leafpos[s]] = sorted[s];
}

template <typename T>
struct DevBuf {
    T* p = nullptr;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t alloc(size_t n) { return cudaMalloc((void**)&p, (n ? n : 1) * sizeof(T)); }
    void release() { if (p) cudaFree(p); p = nullptr; }
};


// ---------------------------------------------------------------- binned SAH, top-down, level-synchronous (the default hierarchy)
// Wald 2007 ("On fast construction of SAH-based bounding volume hierarchies"), run breadth-first on the device: every open
// subtree of a level is an ITEM; per level
//   k_sah_bin       every triangle adds its box to one of SAH_BINS bins per axis of its item (integer atomics on ordered floats)
//   k_sah_split     one thread per item: box -> the parent's node, sweep the 3 x 16 bins, leaf or split
//   (exclusive scan of the split flags: inner-node numbers and next level's item slots, deterministic)
//   k_sah_children  split items name their inner node and open two items in the next level
//   k_sah_assign    every triangle moves to its child item (and adds itself to that item's bounds) or records its leaf
// One read-back per level (the number of splits).  Triangles are never moved: a leaf's first slot in leaf order is known from
// the counts on the way down (left subtree first), and ONE stable radix sort by that slot at the end gives the leaf order.
// Every atomic is an integer min / max / add, so the tree is identical from run to run.
// Traversal time of flying_unicorn against PLOC: -8 % (tools/gpu_bvh_quality.py); a full-sweep SAH on the host gains 1 % more.
constexpr int SAH_BINS = 16;
constexpr float SAH_NODE_COST = 1.0f;    // one node visit in units of one triangle test (flat between 0.7 and 2)

struct SahItem {
    int lo[3], hi[3], clo[3], chi[3];   // triangle / centroid bounds, ordered ints (same layout as Bounds6)
    int count;
    int imin, imax;                     // triangle index range: splits a subtree whose centroids all coincide
    int parent2;                        // inner node that owns this item * 2 + side; -1: the root
    int first_base;                     // first leaf-order slot of the PARENT's range
};
struct SahBin { int lo[3], hi[3], count; };
struct SahDecision { int kind, axis, split, first; };   // kind 0 leaf, 1 split after bin `split` of `axis`, 2 split at triangle index `split`

__device__ __forceinline__ int sah_bin_of(float c, float clo, float ext) {
    return min(SAH_BINS - 1, max(0, (int)((c - clo) * ((float)SAH_BINS / ext))));
}
__device__ __forceinline__ float sah_area(const int* lo, const int* hi) {
    float dx = ordered_to_float(hi[0]) - ordered_to_float(lo[0]), dy = ordered_to_float(hi[1]) - ordered_to_float(lo[1]),
          dz = ordered_to_float(hi[2]) - ordered_to_float(lo[2]);
    return dx * dy + dy * dz + dz * dx;
}

__global__ void k_sah_root(const Bounds6* gb, int n, SahItem* items, int* item_of) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) item_of[i] = 0;
    if (i == 0) {
        SahItem it;
        for (int k = 0; k < 3; ++k) { it.lo[k] = gb->lo[k]; it.hi[k] = gb->hi[k]; it.clo[k] = gb->clo[k]; it.chi[k] = gb->chi[k]; }
        it.count = n; it.imin = 0; it.imax = n - 1; it.parent2 = -1; it.first_base = 0;
        items[0] = it;
    }
}

__global__ void k_sah_clear_bins(int nbins, SahBin* bins) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nbins) return;
    SahBin b;
    for (int k = 0; k < 3; ++k) { b.lo[k] = float_to_ordered(FLT_MAX); b.hi[k] = float_to_ordered(-FLT_MAX); }
    b.count = 0;
    bins[i] = b;
}

__global__ void k_sah_bin(int n, const int* __restrict__ item_of, const SahItem* __restrict__ items, const float4* __restrict__ tlo,
                          const float4* __restrict__ thi, SahBin* bins) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = item_of[i];
    if (j < 0) return;
    const SahItem& it = items[j];
    if (it.count < 2) return;
    const float4 lo = tlo[i], hi = thi[i];
    const float c[3] = {0.5f * (lo.x + hi.x), 0.5f * (lo.y + hi.y), 0.5f * (lo.z + hi.z)};
    const int olo[3] = {float_to_ordered(lo.x), float_to_ordered(lo.y), float_to_ordered(lo.z)};
    const int ohi[3] = {float_to_ordered(hi.x), float_to_ordered(hi.y), float_to_ordered(hi.z)};
    for (int ax = 0; ax < 3; ++ax) {
        const float clo = ordered_to_float(it.clo[ax]), ext = ordered_to_float(it.chi[ax]) - clo;
        if (!(ext > 0.f)) continue;
        SahBin* b = bins + ((size_t)j * 3 + ax) * SAH_BINS + sah_bin_of(c[ax], clo, ext);
        for (int k = 0; k < 3; ++k) { atomicMin(&b->lo[k], olo[k]); atomicMax(&b->hi[k], ohi[k]); }
        atomicAdd(&b->count, 1);
    }
}

__global__ void k_sah_split(int m, const SahItem* __restrict__ items, const SahBin* __restrict__ bins, int leaf_max, float node_cost,
                            float4* __restrict__ nodes, int* root_ref, SahDecision* __restrict__ dec, int* __restrict__ flag) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m) return;
    const SahItem& it = items[j];
    const int side = it.parent2 & 1, parent = it.parent2 >> 1;
    const int first = it.first_base + ((it.parent2 >= 0 && side) ? items[j - 1].count : 0);
    if (it.parent2 >= 0) {   // this subtree's box, into its slot of the parent's node
        float* o = reinterpret_cast<float*>(nodes + (size_t)parent * 4);
        o[side * 4 + 0] = ordered_to_float(it.lo[0]); o[side * 4 + 1] = ordered_to_float(it.hi[0]);
        o[side * 4 + 2] = ordered_to_float(it.lo[1]); o[side * 4 + 3] = ordered_to_float(it.hi[1]);
        o[8 + side * 2 + 0] = ordered_to_float(it.lo[2]); o[8 + side * 2 + 1] = ordered_to_float(it.hi[2]);
    }
    float best = FLT_MAX;
    int bax = -1, bsplit = -1;
    if (it.count >= 2) {
        for (int ax = 0; ax < 3; ++ax) {
            if (!(ordered_to_float(it.chi[ax]) - ordered_to_float(it.clo[ax]) > 0.f)) continue;
            const SahBin* b = bins + ((size_t)j * 3 + ax) * SAH_BINS;
            float ra[SAH_BINS];
            int alo[3], ahi[3];
            for (int k = 0; k < 3; ++k) { alo[k] = float_to_ordered(FLT_MAX); ahi[k] = float_to_ordered(-FLT_MAX); }
            for (int q = SAH_BINS - 1; q > 0; --q) {
                if (b[q].count) for (int k = 0; k < 3; ++k) { alo[k] = min(alo[k], b[q].lo[k]); ahi[k] = max(ahi[k], b[q].hi[k]); }
                ra[q] = sah_area(alo, ahi);
            }
            for (int k = 0; k < 3; ++k) { alo[k] = float_to_ordered(FLT_MAX); ahi[k] = float_to_ordered(-FLT_MAX); }
            int lc = 0;
            for (int q = 0; q < SAH_BINS - 1; ++q) {
                if (b[q].count) for (int k = 0; k < 3; ++k) { alo[k] = min(alo[k], b[q].lo[k]); ahi[k] = max(ahi[k], b[q].hi[k]); }
                lc += b[q].count;
                const int rc = it.count - lc;
                if (lc == 0 || rc == 0) continue;
                const float cost = sah_area(alo, ahi) * (float)lc + ra[q + 1] * (float)rc;
                if (cost < best) { best = cost; bax = ax; bsplit = q; }
            }
        }
    }
    const float A = sah_area(it.lo, it.hi);
    SahDecision d;
    d.first = first;
    d.axis = bax;
    d.split = bsplit;
    if (it.count < 2 || (it.count <= leaf_max && (bax < 0 || node_cost * A + best >= A * (float)it.count)) || (bax < 0 && it.count <= 8)) d.kind = 0;
    else if (bax < 0) { d.kind = 2; d.split = it.imin + (it.imax - it.imin) / 2; }   // coinciding centroids: halve the index range
    else d.kind = 1;
    dec[j] = d;
    flag[j] = d.kind != 0;
    if (d.kind == 0) {
        const int ref = encode_leaf(first, it.count);
        if (it.parent2 >= 0) reinterpret_cast<int*>(nodes + (size_t)parent * 4 + 3)[side] = ref;
        else *root_ref = ref;
    }
}

__global__ void k_sah_children(int m, const SahItem* __restrict__ items, const SahDecision* __restrict__ dec, const int* __restrict__ flag,
                               const int* __restrict__ pos, int inner_base, float4* __restrict__ nodes, int* root_ref, SahItem* __restrict__ next) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= m || !flag[j]) return;
    const SahItem& it = items[j];
    const int inner = inner_base + pos[j];
    if (it.parent2 >= 0) reinterpret_cast<int*>(nodes + (size_t)(it.parent2 >> 1) * 4 + 3)[it.parent2 & 1] = inner;
    else *root_ref = inner;
    reinterpret_cast<int*>(nodes + (size_t)inner * 4 + 3)[2] = 0;
    reinterpret_cast<int*>(nodes + (size_t)inner * 4 + 3)[3] = 0;
    for (int s = 0; s < 2; ++s) {
        SahItem c;
        for (int k = 0; k < 3; ++k) {
            c.lo[k] = c.clo[k] = float_to_ordered(FLT_MAX);
            c.hi[k] = c.chi[k] = float_to_ordered(-FLT_MAX);
        }
        c.count = 0; c.imin = 0x7fffffff; c.imax = -1;
        c.parent2 = inner * 2 + s;
        c.first_base = dec[j].first;
        next[2 * pos[j] + s] = c;
    }
}

__global__ void k_sah_assign(int n, int* __restrict__ item_of, const SahItem* __restrict__ items, const SahDecision* __restrict__ dec,
                             const int* __restrict__ pos, const float4* __restrict__ tlo, const float4* __restrict__ thi, SahItem* next,
                             uint32_t* __restrict__ leaf_slot) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int j = item_of[i];
    if (j < 0) return;
    const SahDecision d = dec[j];
    if (d.kind == 0) {
        leaf_slot[i] = (uint32_t)d.first;
        item_of[i] = -1;
        return;
    }
    const float4 lo = tlo[i], hi = thi[i];
    const float c[3] = {0.5f * (lo.x + hi.x), 0.5f * (lo.y + hi.y), 0.5f * (lo.z + hi.z)};
    int side;
    if (d.kind == 1) {
        const float clo = ordered_to_float(items[j].clo[d.axis]), ext = ordered_to_float(items[j].chi[d.axis]) - clo;
        side = sah_bin_of(c[d.axis], clo, ext) > d.split;
    } else side = i > d.split;
    const int nj = 2 * pos[j] + side;
    SahItem* t = next + nj;
    atomicMin(&t->lo[0], float_to_ordered(lo.x)); atomicMin(&t->lo[1], float_to_ordered(lo.y)); atomicMin(&t->lo[2], float_to_ordered(lo.z));
    atomicMax(&t->hi[0], float_to_ordered(hi.x)); atomicMax(&t->hi[1], float_to_ordered(hi.y)); atomicMax(&t->hi[2], float_to_ordered(hi.z));
    for (int k = 0; k < 3; ++k) { atomicMin(&t->clo[k], float_to_ordered(c[k])); atomicMax(&t->chi[k], float_to_ordered(c[k])); }
    atomicAdd(&t->count, 1);
    atomicMin(&t->imin, i);
    atomicMax(&t->imax, i);
    item_of[i] = nj;
}

__global__ void k_iota(int n, uint32_t* v) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = (uint32_t)i;
}

}  // namespace

// ---- DIAGNOSTIC (RTB_BVH=sah_host): host-side SAH build into the same node format — the prototype the device builder above was
// checked against (same policy by default: 16 bins, leaves of <= 2 triangles, node cost 1 -> the same node count), with knobs the
// device builder does not have (RTB_SAH_BINS, RTB_SAH_SWEEP = full sweep below that many triangles, RTB_SAH_LEAF, RTB_SAH_CT).
// Not the product path.
namespace {
struct HB { float lo[3], hi[3]; };
struct SahBuilder {
    const float* v; int n;
    std::vector<HB> tb; std::vector<float> cen;   // per triangle
    std::vector<int> order;
    std::vector<float4> nodes;                    // 4 per node
    static float area(const HB& b) { float dx=b.hi[0]-b.lo[0], dy=b.hi[1]-b.lo[1], dz=b.hi[2]-b.lo[2]; return 2.f*(dx*dy+dy*dz+dz*dx); }
    static void grow(HB& a, const HB& b) { for (int k=0;k<3;++k){ a.lo[k]=fminf(a.lo[k],b.lo[k]); a.hi[k]=fmaxf(a.hi[k],b.hi[k]); } }
    static HB empty() { HB b; for (int k=0;k<3;++k){ b.lo[k]=FLT_MAX; b.hi[k]=-FLT_MAX; } return b; }
    int nbins = 16, sweep_max = 0, leaf_max = 2;
    float ct = 1.f;                                  // cost of one node visit in units of one triangle test (= SAH_NODE_COST)
    std::vector<float> ra_s;                         // sweep scratch
    // returns encoded ref (>=0 node, <0 leaf) and the box
    int build(int first, int count, HB& box) {
        box = empty();
        HB cb = empty();
        for (int i=first;i<first+count;++i){ int t=order[i]; grow(box,tb[t]); for(int k=0;k<3;++k){ cb.lo[k]=fminf(cb.lo[k],cen[3*t+k]); cb.hi[k]=fmaxf(cb.hi[k],cen[3*t+k]); } }
        if (count == 1) return ~((first << 3) | 0);
        float best = FLT_MAX; int bax=-1, bsplit=-1; bool swept = false;
        if (count <= sweep_max) {                    // full sweep: every split position of every axis
            swept = true;
            ra_s.resize(count);
            for (int ax=0; ax<3; ++ax) {
                std::sort(order.begin()+first, order.begin()+first+count, [&](int a, int b){ float ca=cen[3*a+ax], cb2=cen[3*b+ax]; return ca<cb2 || (ca==cb2 && a<b); });
                HB acc=empty();
                for (int i=count-1;i>0;--i){ grow(acc,tb[order[first+i]]); ra_s[i]=area(acc); }
                acc=empty();
                for (int i=0;i<count-1;++i){ grow(acc,tb[order[first+i]]); float cost=area(acc)*(i+1)+ra_s[i+1]*(count-i-1); if(cost<best){best=cost;bax=ax;bsplit=i+1;} }
            }
            if (bax >= 0 && bax != 2) std::sort(order.begin()+first, order.begin()+first+count, [&](int a, int b){ float ca=cen[3*a+bax], cb2=cen[3*b+bax]; return ca<cb2 || (ca==cb2 && a<b); });
        } else {
            const int NB = nbins;
            for (int ax=0; ax<3; ++ax) {
                float ext = cb.hi[ax]-cb.lo[ax];
                if (!(ext > 0.f)) continue;
                HB bb[64]; int bc[64];
                for (int b=0;b<NB;++b){ bb[b]=empty(); bc[b]=0; }
                for (int i=first;i<first+count;++i){ int t=order[i]; int b=(int)((cen[3*t+ax]-cb.lo[ax])/ext*NB); if(b>=NB)b=NB-1; if(b<0)b=0; grow(bb[b],tb[t]); bc[b]++; }
                float ra[64]; HB acc=empty();
                for (int b=NB-1;b>0;--b){ grow(acc,bb[b]); ra[b]=area(acc); }
                acc=empty(); int lc=0; int rc=count;
                for (int b=0;b<NB-1;++b){ grow(acc,bb[b]); lc+=bc[b]; rc=count-lc; if(lc==0||rc==0) continue; float cost=area(acc)*lc+ra[b+1]*rc; if(cost<best){best=cost;bax=ax;bsplit=b;} }
            }
        }
        const float leaf_cost = area(box) * count;
        if (count <= leaf_max && (bax < 0 || ct * area(box) + best >= leaf_cost)) return ~((first << 3) | (count - 1));
        int mid;
        if (bax < 0) {
            if (count <= 8) return ~((first << 3) | (count - 1));
            mid = first + count/2;                   // degenerate: median split on order
        } else if (swept) mid = first + bsplit;
        else {
            const int NB = nbins;
            float ext = cb.hi[bax]-cb.lo[bax];
            mid = (int)(std::partition(order.begin()+first, order.begin()+first+count, [&](int t){ int b=(int)((cen[3*t+bax]-cb.lo[bax])/ext*NB); if(b>=NB)b=NB-1; if(b<0)b=0; return b<=bsplit; }) - order.begin());
            if (mid==first || mid==first+count) mid = first+count/2;
        }
        int idx=(int)nodes.size()/4; nodes.resize(nodes.size()+4);
        HB lb, rb;
        int l = build(first, mid-first, lb), r = build(mid, first+count-mid, rb);
        emit(idx, l, r, lb, rb);
        return idx;
    }
    void emit(int idx, int l, int r, const HB& a, const HB& b) {
        float4* o = &nodes[(size_t)idx*4];
        o[0]=make_float4(a.lo[0],a.hi[0],a.lo[1],a.hi[1]);
        o[1]=make_float4(b.lo[0],b.hi[0],b.lo[1],b.hi[1]);
        o[2]=make_float4(a.lo[2],a.hi[2],b.lo[2],b.hi[2]);
        int li=l, ri=r; float fl, fr; memcpy(&fl,&li,4); memcpy(&fr,&ri,4);
        o[3]=make_float4(fl,fr,0.f,0.f);
    }
};
}  // namespace

static bool build_sah_host(const float* d_verts, const int32_t* d_tri_obj, int n, cudaStream_t stream, LbvhResult& out, std::string& err) {
    std::vector<float> hv((size_t)n*9);
    LBVH_CHECK(cudaMemcpyAsync(hv.data(), d_verts, hv.size()*sizeof(float), cudaMemcpyDeviceToHost, stream));
    LBVH_CHECK(cudaStreamSynchronize(stream));
    SahBuilder B; B.v=hv.data(); B.n=n; B.tb.resize(n); B.cen.resize((size_t)3*n); B.order.resize(n);
    HB all=SahBuilder::empty();
    for (int i=0;i<n;++i){ HB b=SahBuilder::empty(); for(int k=0;k<3;++k){ for(int q=0;q<3;++q){ float x=hv[(size_t)i*9+3*q+k]; b.lo[k]=fminf(b.lo[k],x); b.hi[k]=fmaxf(b.hi[k],x);} float pad=fmaxf(fabsf(b.lo[k]),fabsf(b.hi[k]))*1e-6f+1e-30f; b.lo[k]-=pad; b.hi[k]+=pad; B.cen[3*i+k]=0.5f*(b.lo[k]+b.hi[k]); } B.tb[i]=b; SahBuilder::grow(all,b); B.order[i]=i; }
    if (const char* e = getenv("RTB_SAH_BINS")) B.nbins = std::min(64, std::max(2, atoi(e)));
    if (const char* e = getenv("RTB_SAH_SWEEP")) B.sweep_max = std::max(0, atoi(e));
    if (const char* e = getenv("RTB_SAH_LEAF")) B.leaf_max = std::min(8, std::max(1, atoi(e)));
    if (const char* e = getenv("RTB_SAH_CT")) B.ct = (float)atof(e);
    HB rootbox; int root = B.build(0, n, rootbox);
    std::vector<uint32_t> ord(B.order.begin(), B.order.end());
    uint32_t* d_ord=nullptr;
    LBVH_CHECK(cudaMalloc((void**)&d_ord, (size_t)n*4));
    LBVH_CHECK(cudaMemcpyAsync(d_ord, ord.data(), (size_t)n*4, cudaMemcpyHostToDevice, stream));
    LBVH_CHECK(cudaMalloc((void**)&out.d_tris, (size_t)n*rtb::TRI_STRIDE*sizeof(float4)));
    LBVH_CHECK(cudaMalloc((void**)&out.d_tri_nrm, (size_t)n*sizeof(float4)));
    k_pack_tris<<<(n+255)/256, 256, 0, stream>>>(n, d_ord, d_verts, d_tri_obj, out.d_tris, out.d_tri_nrm);
    out.n_nodes=(int)B.nodes.size()/4;
    LBVH_CHECK(cudaMalloc((void**)&out.d_nodes, (size_t)(out.n_nodes?out.n_nodes:1)*4*sizeof(float4)));
    if (out.n_nodes) LBVH_CHECK(cudaMemcpyAsync(out.d_nodes, B.nodes.data(), B.nodes.size()*sizeof(float4), cudaMemcpyHostToDevice, stream));
    LBVH_CHECK(cudaStreamSynchronize(stream));
    cudaFree(d_ord);
    out.root=root; out.n_leaves=out.n_nodes+1;
    for (int k=0;k<3;++k){ out.bmin[k]=all.lo[k]; out.bmax[k]=all.hi[k]; }
    return true;
}

// 64-byte fp32 nodes -> 32-byte nodes for the traversal kernels, which are bound by the L1 data pipe (one wavefront per
// divergent lane and load instruction): ONE 256-bit load per node visit instead of two.
//   word 0..2: child 0 (lo.x | hi.x << 16), (lo.y | hi.y << 16), (lo.z | hi.z << 16)     word 3..5: child 1     word 6, 7: child references
// A box coordinate k stands for the plane qmin + k * qstep (qstep = extent of all triangles / 65535).  lo is rounded down and hi
// up, plus QPAD steps: the traversal rebuilds the slab distances with one FMA per plane from the integer (8388608 + k), whose
// rounding moves a plane by at most one step (see trav_begin), and uses approximate reciprocals.
constexpr int QPAD = 2;
__global__ void k_quantise_nodes(int n_nodes, const float4* __restrict__ nodes, uint4* __restrict__ out, float3 qmin, float3 qinv) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_nodes) return;
    const float4 n0 = nodes[(size_t)i * 4], n1 = nodes[(size_t)i * 4 + 1], n2 = nodes[(size_t)i * 4 + 2], n3 = nodes[(size_t)i * 4 + 3];
    auto qlo = [](float v, float m, float inv) { int k = (int)floorf((v - m) * inv) - QPAD; return (uint32_t)min(max(k, 0), 65535); };
    auto qhi = [](float v, float m, float inv) { int k = (int)ceilf((v - m) * inv) + QPAD; return (uint32_t)min(max(k, 0), 65535); };
    uint4 a, b;
    a.x = qlo(n0.x, qmin.x, qinv.x) | (qhi(n0.y, qmin.x, qinv.x) << 16);
    a.y = qlo(n0.z, qmin.y, qinv.y) | (qhi(n0.w, qmin.y, qinv.y) << 16);
    a.z = qlo(n2.x, qmin.z, qinv.z) | (qhi(n2.y, qmin.z, qinv.z) << 16);
    a.w = qlo(n1.x, qmin.x, qinv.x) | (qhi(n1.y, qmin.x, qinv.x) << 16);
    b.x = qlo(n1.z, qmin.y, qinv.y) | (qhi(n1.w, qmin.y, qinv.y) << 16);
    b.y = qlo(n2.z, qmin.z, qinv.z) | (qhi(n2.w, qmin.z, qinv.z) << 16);
    b.z = __float_as_uint(n3.x);
    b.w = __float_as_uint(n3.y);
    out[(size_t)i * 2] = a;
    out[(size_t)i * 2 + 1] = b;
}

static bool build_lbvh_f32(const float* d_verts, const int32_t* d_tri_obj, int n, cudaStream_t stream, LbvhResult& out, std::string& err,
                           bool force_karras = false);

// Depth of the binary tree: 0 when the root is a leaf, otherwise the root is level 1 and every inner child one more.  The
// traversal stack is finite: build_lbvh checks it against BVH_MAX_DEPTH.  Walked on the host over the finished fp32 table.
static bool measure_depth(cudaStream_t stream, LbvhResult& out, std::string& err) {
    out.depth = 0;
    if (out.n_nodes == 0 || out.root < 0) return true;
    std::vector<float4> nodes((size_t)out.n_nodes * 4);
    LBVH_CHECK(cudaMemcpyAsync(nodes.data(), out.d_nodes, nodes.size() * sizeof(float4), cudaMemcpyDeviceToHost, stream));
    LBVH_CHECK(cudaStreamSynchronize(stream));
    std::vector<std::pair<int, int>> st;
    st.push_back({out.root, 1});
    while (!st.empty()) {
        const auto [node, d] = st.back();
        st.pop_back();
        out.depth = std::max(out.depth, d);
        int ref[2];
        memcpy(ref, &nodes[(size_t)node * 4 + 3].x, sizeof(ref));   // float4 3 of the node: (ref 0, ref 1, -, -)
        for (int k = 0; k < 2; ++k)
            if (ref[k] >= 0) st.push_back({ref[k], d + 1});
    }
    return true;
}

static bool build_lbvh_tables(const float* d_verts, const int32_t* d_tri_obj, int n, cudaStream_t stream, LbvhResult& out, std::string& err,
                              bool force_karras) {
    if (!build_lbvh_f32(d_verts, d_tri_obj, n, stream, out, err, force_karras)) return false;
    if (n <= 0) return true;
    float3 qinv;
    float* qi = &qinv.x;
    for (int k = 0; k < 3; ++k) {
        const float ext = fmaxf(out.bmax[k] - out.bmin[k], 1e-20f);
        out.qmin[k] = out.bmin[k];
        out.qstep[k] = ext / 65535.0f;
        qi[k] = 65535.0f / ext;
    }
    LBVH_CHECK(cudaMalloc((void**)&out.d_qnodes, (size_t)(out.n_nodes ? out.n_nodes : 1) * 2 * sizeof(uint4)));
    if (out.n_nodes) {
        k_quantise_nodes<<<(out.n_nodes + 255) / 256, 256, 0, stream>>>(out.n_nodes, out.d_nodes, out.d_qnodes,
                                                                      make_float3(out.qmin[0], out.qmin[1], out.qmin[2]), qinv);
        LBVH_CHECK(cudaStreamSynchronize(stream));
        LBVH_CHECK(cudaGetLastError());
    }
    return measure_depth(stream, out, err);
}

// The traversal stack holds BVH_MAX_DEPTH levels.  A Karras tree over 63-bit keys + a 32-bit tie-break cannot be deeper
// than 95; a PLOC tree has no such bound (a chain of single mutual-pair merges adds one level per round), so a PLOC tree
// that came out too deep is rebuilt with the Karras hierarchy, and a mesh whose tree still does not fit is refused
// ("unsupported: ..." -> RTB_EUNSUPPORTED) instead of being traversed with an overflowing stack.
bool build_lbvh(const float* d_verts, const int32_t* d_tri_obj, int n, cudaStream_t stream, LbvhResult& out, std::string& err) {
    const int max_depth = depth_limit();
    if (!build_lbvh_tables(d_verts, d_tri_obj, n, stream, out, err, false)) return false;
    if (out.depth > max_depth) {
        free_lbvh(out);
        if (!build_lbvh_tables(d_verts, d_tri_obj, n, stream, out, err, true)) return false;
    }
    if (out.depth > max_depth) {
        err = "unsupported: the mesh's BVH is " + std::to_string(out.depth) + " levels deep, the traversal stack holds " + std::to_string(max_depth);
        free_lbvh(out);
        return false;
    }
    return true;
}

static bool build_lbvh_f32(const float* d_verts, const int32_t* d_tri_obj, int n, cudaStream_t stream, LbvhResult& out, std::string& err,
                           bool force_karras) {
    out = LbvhResult();
    if (n <= 0) return true;
    const std::string mode = getenv("RTB_BVH") ? getenv("RTB_BVH") : "";
    if (!force_karras && mode == "sah_host") return build_sah_host(d_verts, d_tri_obj, n, stream, out, err);
    const int T = 256;
    const int nb = (n + T - 1) / T;
    const int ni = n - 1;

    DevBuf<float4> tlo, thi, nlo, nhi;
    DevBuf<Bounds6> gb;
    DevBuf<unsigned long long> keys, keys2;
    DevBuf<uint32_t> vals, vals2;
    DevBuf<int> left, right, pint, pleaf, rfirst, rlast, arrive, used, newidx;
    LBVH_CHECK(tlo.alloc(n)); LBVH_CHECK(thi.alloc(n)); LBVH_CHECK(nlo.alloc(n)); LBVH_CHECK(nhi.alloc(n));
    LBVH_CHECK(gb.alloc(1));
    LBVH_CHECK(keys.alloc(n)); LBVH_CHECK(keys2.alloc(n)); LBVH_CHECK(vals.alloc(n)); LBVH_CHECK(vals2.alloc(n));
    LBVH_CHECK(left.alloc(n)); LBVH_CHECK(right.alloc(n)); LBVH_CHECK(pint.alloc(n)); LBVH_CHECK(pleaf.alloc(n));
    LBVH_CHECK(rfirst.alloc(n)); LBVH_CHECK(rlast.alloc(n)); LBVH_CHECK(arrive.alloc(n)); LBVH_CHECK(used.alloc(n));
    LBVH_CHECK(newidx.alloc(n + 1));

    k_init_bounds<<<1, 1, 0, stream>>>(gb.p);
    k_tri_bounds<<<nb, T, 0, stream>>>(d_verts, n, tlo.p, thi.p, gb.p);
    const bool karras = force_karras || mode == "lbvh";
    const bool sah = !karras && mode != "ploc" && n > LEAF_MAX;   // default: binned SAH, top-down; "ploc" / "lbvh": bottom-up over the Morton order
    k_morton<<<nb, T, 0, stream>>>(tlo.p, thi.p, n, gb.p, keys.p, vals.p);

    size_t tmp_bytes = 0, scan_bytes = 0;
    LBVH_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys.p, keys2.p, vals.p, vals2.p, n, 0, 63, stream));
    LBVH_CHECK(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, used.p, newidx.p, n, stream));
    DevBuf<unsigned char> tmp;
    LBVH_CHECK(tmp.alloc(tmp_bytes > scan_bytes ? tmp_bytes : scan_bytes));
    if (!sah) LBVH_CHECK(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, keys.p, keys2.p, vals.p, vals2.p, n, 0, 63, stream));   // the SAH builder has no use for the Morton order

    float4* d_tris = nullptr;
    LBVH_CHECK(cudaMalloc((void**)&d_tris, (size_t)n * rtb::TRI_STRIDE * sizeof(float4)));
    out.d_tris = d_tris;
    LBVH_CHECK(cudaMalloc((void**)&out.d_tri_nrm, (size_t)n * sizeof(float4)));

    Bounds6 hb;
    int leaf_max = LEAF_MAX;
    if (const char* e = getenv("RTB_LEAF_MAX")) leaf_max = std::min(8, std::max(1, atoi(e)));
    if (n <= LEAF_MAX) {  // the whole mesh is one leaf
        k_pack_tris<<<nb, T, 0, stream>>>(n, vals2.p, d_verts, d_tri_obj, d_tris, out.d_tri_nrm);
        out.root = ~((0 << 3) | (n - 1));
        out.n_nodes = 0;
        out.n_leaves = 1;
        LBVH_CHECK(cudaMalloc((void**)&out.d_nodes, 4 * sizeof(float4)));
    } else if (karras) {
        k_pack_tris<<<nb, T, 0, stream>>>(n, vals2.p, d_verts, d_tri_obj, d_tris, out.d_tri_nrm);
        LBVH_CHECK(cudaMemsetAsync(arrive.p, 0, (size_t)n * sizeof(int), stream));
        const int nbi = (ni + T - 1) / T;
        k_hierarchy<<<nbi, T, 0, stream>>>(keys2.p, n, left.p, right.p, pint.p, pleaf.p, rfirst.p, rlast.p);
        k_refit<<<nb, T, 0, stream>>>(n, vals2.p, tlo.p, thi.p, left.p, right.p, pint.p, pleaf.p, arrive.p, nlo.p, nhi.p);
        k_mark_used<<<nbi, T, 0, stream>>>(ni, leaf_max, rfirst.p, rlast.p, used.p);
        LBVH_CHECK(cub::DeviceScan::ExclusiveSum(tmp.p, scan_bytes, used.p, newidx.p, ni, stream));
        int last_used = 0, last_idx = 0;
        LBVH_CHECK(cudaMemcpyAsync(&last_used, used.p + (ni - 1), sizeof(int), cudaMemcpyDeviceToHost, stream));
        LBVH_CHECK(cudaMemcpyAsync(&last_idx, newidx.p + (ni - 1), sizeof(int), cudaMemcpyDeviceToHost, stream));
        LBVH_CHECK(cudaStreamSynchronize(stream));
        out.n_nodes = last_idx + last_used;
        LBVH_CHECK(cudaMalloc((void**)&out.d_nodes, (size_t)(out.n_nodes ? out.n_nodes : 1) * 4 * sizeof(float4)));
        k_emit<<<nbi, T, 0, stream>>>(ni, vals2.p, tlo.p, thi.p, left.p, right.p, rfirst.p, rlast.p, used.p, newidx.p, nlo.p,
                                      nhi.p, out.d_nodes, nullptr);
        out.root = 0;  // Karras: internal node 0 is the root; it is always used here (n > LEAF_MAX) and keeps index 0
        out.n_leaves = out.n_nodes + 1;
    } else if (sah) {
        DevBuf<SahItem> items[2];
        DevBuf<SahBin> bins;
        DevBuf<SahDecision> dec;
        DevBuf<int> flag, pos, item_of, root_ref;
        DevBuf<uint32_t> slot, slot2, ids, order;
        DevBuf<unsigned char> tmp2;
        LBVH_CHECK(items[0].alloc(n)); LBVH_CHECK(items[1].alloc(n)); LBVH_CHECK(dec.alloc(n)); LBVH_CHECK(flag.alloc(n)); LBVH_CHECK(pos.alloc(n + 1));
        LBVH_CHECK(item_of.alloc(n)); LBVH_CHECK(root_ref.alloc(1)); LBVH_CHECK(slot.alloc(n)); LBVH_CHECK(slot2.alloc(n)); LBVH_CHECK(ids.alloc(n));
        LBVH_CHECK(order.alloc(n));
        LBVH_CHECK(cudaMalloc((void**)&out.d_nodes, (size_t)n * 4 * sizeof(float4)));   // at most n - 1 inner nodes
        size_t bins_cap = 0;
        k_sah_root<<<nb, T, 0, stream>>>(gb.p, n, items[0].p, item_of.p);
        int m = 1, inner = 0, cur = 0, levels = 0;
        while (m > 0) {
            if (++levels > depth_limit() + 1) {   // already deeper than the traversal stack holds (16 bins peel at least one exponent
                free_lbvh(out);                   // step of centroid range per level, so this takes an adversarial mesh): Karras' turn
                return build_lbvh_f32(d_verts, d_tri_obj, n, stream, out, err, true);
            }
            const size_t nbins = (size_t)m * 3 * SAH_BINS;
            if (nbins > bins_cap) {
                LBVH_CHECK(cudaStreamSynchronize(stream));
                bins.release();
                bins_cap = std::max(nbins, 2 * bins_cap);
                LBVH_CHECK(bins.alloc(bins_cap));
            }
            const int mb = (m + T - 1) / T;
            k_sah_clear_bins<<<(int)((nbins + T - 1) / T), T, 0, stream>>>((int)nbins, bins.p);
            k_sah_bin<<<nb, T, 0, stream>>>(n, item_of.p, items[cur].p, tlo.p, thi.p, bins.p);
            k_sah_split<<<mb, T, 0, stream>>>(m, items[cur].p, bins.p, leaf_max, SAH_NODE_COST, out.d_nodes, root_ref.p, dec.p, flag.p);
            LBVH_CHECK(cub::DeviceScan::ExclusiveSum(tmp.p, scan_bytes, flag.p, pos.p, m, stream));
            k_sah_children<<<mb, T, 0, stream>>>(m, items[cur].p, dec.p, flag.p, pos.p, inner, out.d_nodes, root_ref.p, items[cur ^ 1].p);
            k_sah_assign<<<nb, T, 0, stream>>>(n, item_of.p, items[cur].p, dec.p, pos.p, tlo.p, thi.p, items[cur ^ 1].p, slot.p);
            int tail[2];  // flag[m-1], pos[m-1]
            LBVH_CHECK(cudaMemcpyAsync(&tail[0], flag.p + (m - 1), sizeof(int), cudaMemcpyDeviceToHost, stream));
            LBVH_CHECK(cudaMemcpyAsync(&tail[1], pos.p + (m - 1), sizeof(int), cudaMemcpyDeviceToHost, stream));
            LBVH_CHECK(cudaStreamSynchronize(stream));
            const int splits = tail[0] + tail[1];
            inner += splits;
            m = 2 * splits;
            cur ^= 1;
        }
        if (inner > n - 1) { err = "SAH node count mismatch"; return false; }
        // leaf order = triangles by the first slot of their leaf (stable: index order inside a leaf)
        size_t sort_bytes = 0;
        k_iota<<<nb, T, 0, stream>>>(n, ids.p);
        LBVH_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, sort_bytes, slot.p, slot2.p, ids.p, order.p, n, 0, 32, stream));
        LBVH_CHECK(tmp2.alloc(sort_bytes));
        LBVH_CHECK(cub::DeviceRadixSort::SortPairs(tmp2.p, sort_bytes, slot.p, slot2.p, ids.p, order.p, n, 0, 32, stream));
        k_pack_tris<<<nb, T, 0, stream>>>(n, order.p, d_verts, d_tri_obj, d_tris, out.d_tri_nrm);
        int root = 0;
        LBVH_CHECK(cudaMemcpyAsync(&root, root_ref.p, sizeof(int), cudaMemcpyDeviceToHost, stream));
        LBVH_CHECK(cudaStreamSynchronize(stream));
        out.root = root;
        out.n_nodes = inner;
        out.n_leaves = inner + 1;
    } else {
        // ---- PLOC: cluster arrays ping-pong between (cn0, cl0, ch0, cs0) and (cn1, ...)
        DevBuf<int> cn[2], cs[2], nnb, valid, merge, pv, pm, nsize, leafpos;
        DevBuf<float4> cl[2], ch[2];
        DevBuf<unsigned char> ir_int, ir_leaf;
        DevBuf<uint32_t> order;
        for (int k = 0; k < 2; ++k) { LBVH_CHECK(cn[k].alloc(n)); LBVH_CHECK(cs[k].alloc(n)); LBVH_CHECK(cl[k].alloc(n)); LBVH_CHECK(ch[k].alloc(n)); }
        LBVH_CHECK(nnb.alloc(n)); LBVH_CHECK(valid.alloc(n)); LBVH_CHECK(merge.alloc(n)); LBVH_CHECK(pv.alloc(n + 1)); LBVH_CHECK(pm.alloc(n + 1));
        LBVH_CHECK(nsize.alloc(n)); LBVH_CHECK(leafpos.alloc(n)); LBVH_CHECK(ir_int.alloc(n)); LBVH_CHECK(ir_leaf.alloc(n)); LBVH_CHECK(order.alloc(n));
        k_ploc_init<<<nb, T, 0, stream>>>(n, vals2.p, tlo.p, thi.p, cn[0].p, cl[0].p, ch[0].p, cs[0].p);
        int ploc_radius = PLOC_RADIUS;
        if (const char* e = getenv("RTB_PLOC_RADIUS")) ploc_radius = std::max(1, atoi(e));
        int m = n, node_base = 0, cur = 0, rounds = 0;
        while (m > 1) {
            const int mb = (m + T - 1) / T;
            k_ploc_nn<<<mb, T, 0, stream>>>(m, ploc_radius, cl[cur].p, ch[cur].p, nnb.p);
            k_ploc_flags<<<mb, T, 0, stream>>>(m, nnb.p, valid.p, merge.p);
            LBVH_CHECK(cub::DeviceScan::ExclusiveSum(tmp.p, scan_bytes, valid.p, pv.p, m, stream));
            LBVH_CHECK(cub::DeviceScan::ExclusiveSum(tmp.p, scan_bytes, merge.p, pm.p, m, stream));
            k_ploc_apply<<<mb, T, 0, stream>>>(m, cn[cur].p, cl[cur].p, ch[cur].p, cs[cur].p, nnb.p, valid.p, merge.p, pv.p, pm.p, node_base,
                                               cn[cur ^ 1].p, cl[cur ^ 1].p, ch[cur ^ 1].p, cs[cur ^ 1].p, left.p, right.p, nlo.p, nhi.p,
                                               nsize.p, pint.p, pleaf.p, ir_int.p, ir_leaf.p);
            int tail[4];  // valid[m-1], pv[m-1], merge[m-1], pm[m-1]
            LBVH_CHECK(cudaMemcpyAsync(&tail[0], valid.p + (m - 1), sizeof(int), cudaMemcpyDeviceToHost, stream));
            LBVH_CHECK(cudaMemcpyAsync(&tail[1], pv.p + (m - 1), sizeof(int), cudaMemcpyDeviceToHost, stream));
            LBVH_CHECK(cudaMemcpyAsync(&tail[2], merge.p + (m - 1), sizeof(int), cudaMemcpyDeviceToHost, stream));
            LBVH_CHECK(cudaMemcpyAsync(&tail[3], pm.p + (m - 1), sizeof(int), cudaMemcpyDeviceToHost, stream));
            LBVH_CHECK(cudaStreamSynchronize(stream));
            const int merges = tail[2] + tail[3];
            if (merges <= 0 || ++rounds > 4096) { err = "PLOC made no progress"; return false; }
            m = tail[0] + tail[1];
            node_base += merges;
            cur ^= 1;
        }
        if (node_base != ni) { err = "PLOC node count mismatch"; return false; }
        const int root_node = ni - 1;   // the last merge
        const int minus1 = -1;
        LBVH_CHECK(cudaMemcpyAsync(pint.p + root_node, &minus1, sizeof(int), cudaMemcpyHostToDevice, stream));
        k_ploc_positions<<<(n + ni + T - 1) / T, T, 0, stream>>>(n, ni, left.p, nsize.p, pint.p, pleaf.p, ir_int.p, ir_leaf.p, leafpos.p,
                                                                rfirst.p, rlast.p);
        k_ploc_order<<<nb, T, 0, stream>>>(n, vals2.p, leafpos.p, order.p);
        k_pack_tris<<<nb, T, 0, stream>>>(n, order.p, d_verts, d_tri_obj, d_tris, out.d_tri_nrm);
        const int nbi = (ni + T - 1) / T;
        k_mark_used<<<nbi, T, 0, stream>>>(ni, leaf_max, rfirst.p, rlast.p, used.p);
        LBVH_CHECK(cub::DeviceScan::ExclusiveSum(tmp.p, scan_bytes, used.p, newidx.p, ni, stream));
        int last_used = 0, last_idx = 0, root_new = 0;
        LBVH_CHECK(cudaMemcpyAsync(&last_used, used.p + (ni - 1), sizeof(int), cudaMemcpyDeviceToHost, stream));
        LBVH_CHECK(cudaMemcpyAsync(&last_idx, newidx.p + (ni - 1), sizeof(int), cudaMemcpyDeviceToHost, stream));
        LBVH_CHECK(cudaMemcpyAsync(&root_new, newidx.p + root_node, sizeof(int), cudaMemcpyDeviceToHost, stream));
        LBVH_CHECK(cudaStreamSynchronize(stream));
        out.n_nodes = last_idx + last_used;
        LBVH_CHECK(cudaMalloc((void**)&out.d_nodes, (size_t)(out.n_nodes ? out.n_nodes : 1) * 4 * sizeof(float4)));
        k_emit<<<nbi, T, 0, stream>>>(ni, vals2.p, tlo.p, thi.p, left.p, right.p, rfirst.p, rlast.p, used.p, newidx.p, nlo.p,
                                      nhi.p, out.d_nodes, leafpos.p);
        out.root = root_new;
        out.n_leaves = out.n_nodes + 1;
    }
    LBVH_CHECK(cudaMemcpyAsync(&hb, gb.p, sizeof(hb), cudaMemcpyDeviceToHost, stream));
    LBVH_CHECK(cudaStreamSynchronize(stream));
    LBVH_CHECK(cudaGetLastError());
    for (int k = 0; k < 3; ++k) {
        int lo = hb.lo[k], hi = hb.hi[k];
        float flo, fhi;
        int t = lo >= 0 ? lo : lo ^ 0x7fffffff;
        memcpy(&flo, &t, 4);
        t = hi >= 0 ? hi : hi ^ 0x7fffffff;
        memcpy(&fhi, &t, 4);
        out.bmin[k] = flo;
        out.bmax[k] = fhi;
    }
    return true;
}

void free_lbvh(LbvhResult& r) {
    if (r.d_nodes) cudaFree(r.d_nodes);
    if (r.d_qnodes) cudaFree(r.d_qnodes);
    if (r.d_tris) cudaFree(r.d_tris);
    if (r.d_tri_nrm) cudaFree(r.d_tri_nrm);
    r = LbvhResult();
}

}  // namespace rtb
