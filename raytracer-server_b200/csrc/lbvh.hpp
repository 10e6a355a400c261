// lbvh.hpp — device-built linear BVH (see lbvh.cu).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

namespace rtb {

constexpr int BVH_MAX_DEPTH = 96;   // levels the traversal stack holds (intersect.cuh: STACK_SMEM + STACK_LOCAL)

struct LbvhResult {
    float4* d_nodes = nullptr;  // 4 x float4 per node: c0 (lo.x hi.x lo.y hi.y), c1 (same), (c0.lo.z c0.hi.z c1.lo.z c1.hi.z), refs
    uint4* d_qnodes = nullptr;  // the node table the traversal reads: 2 x uint4 (32 B) per node, child boxes quantised to 16 bits
                                // on the grid qmin + k * qstep (conservative), see quantise_nodes in lbvh.cu
    float qmin[3] = {0, 0, 0}, qstep[3] = {1, 1, 1};
    float4* d_tris = nullptr;   // TRI_STRIDE (4) x float4 per triangle in leaf order: (a | 1/|N|), (b-a | global tri id), (c-a | object id), pad
    float4* d_tri_nrm = nullptr; // 1 x float4 per triangle in leaf order: Triangle::normal (unit) | object id
    int root = 0;               // encoded reference: >= 0 node index, < 0 leaf ~((first << 3) | (count - 1))
    int n_nodes = 0;
    int n_leaves = 0;
    int depth = 0;              // levels of inner nodes on the longest root-to-leaf path (0: the whole mesh is one leaf)
    float bmin[3] = {0, 0, 0}, bmax[3] = {0, 0, 0};
};

// d_verts: 9 floats per triangle (a, b, c) in global triangle order; d_tri_obj: owning object.
bool build_lbvh(const float* d_verts, const int32_t* d_tri_obj, int n, cudaStream_t stream, LbvhResult& out, std::string& err);
void free_lbvh(LbvhResult& r);

}  // namespace rtb
