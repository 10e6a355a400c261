// engine.cu — host runtime of librtb200.so: scene upload, render contexts, the wavefront launch
// loop, streaming jobs and the C ABI declared in include/rtb200.h.
//
// Stands in for the reference's callers of the hot path: Scene::from_toml (src/scene.rs:143-150),
// RenderJob::run (src/server.rs:157-199) and sample_pixel (src/server.rs:320-364).
#include <cuda_runtime.h>

#include <algorithm>
#include <climits>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/rtb200.h"
#include "lbvh.hpp"
#include "octree_host.hpp"
#include "scene_host.hpp"
#include "wavefront.cuh"
#include "denoise.cuh"

using namespace rtb;

namespace {

thread_local std::string g_last_error;
// counters of the calling thread's most recent render call (rtb_get_stats prefers them over the scene-global copy)
thread_local rtb_stats g_thread_stats{};
thread_local const void* g_thread_stats_scene = nullptr;

int fail(int code, const std::string& msg) {
    g_last_error = msg;
    return code;
}

#define CU_TRY(x)                                                                                           \
    do {                                                                                                    \
        cudaError_t e_ = (x);                                                                               \
        if (e_ != cudaSuccess)                                                                              \
            return fail(RTB_ECUDA, std::string(#x) + ": " + cudaGetErrorString(e_) + " (" __FILE__ ":" + std::to_string(__LINE__) + ")"); \
    } while (0)

static_assert(sizeof(FlatPrim) == sizeof(DevPrim), "FlatPrim/DevPrim layout");
static_assert(sizeof(FlatMaterial) == sizeof(DevMaterial), "FlatMaterial/DevMaterial layout");
static_assert(sizeof(DevPrim) == 48 && sizeof(DevMaterial) == 80, "16-byte multiples expected by stage_scene");
static_assert(MAX_OBJECTS == (int)TRI_BASE, "primitive code space");
static_assert(BVH_MAX_DEPTH == STACK_SMEM + STACK_LOCAL, "the loader's depth limit is the traversal stack's capacity");

struct RenderContext {
    int device = 0;
    cudaStream_t stream = nullptr, copy_stream = nullptr;
    bool initialised = false;   // set once the whole one-time set-up below has succeeded
    uint32_t P = 0, SP = 0;         // path / shadow slots of the CURRENT request (logical)
    uint32_t Pcap = 0, SPcap = 0;   // slots the current request addresses: P, SP + room for k_shade's unfilled segment tails
    uint32_t Palloc = 0, SPalloc = 0;   // slots allocated: buffers only ever grow, a smaller request uses the front part
    float4* qbuf = nullptr;      // 2 queues x (4 float4 arrays + 1 float2 array) x P
    float4* sbuf = nullptr;      // 2 shadow queues x 3 arrays x SP
    float4* accum = nullptr;
    size_t accum_cap = 0;
    uint32_t* bin_buf = nullptr;     // coherence binning: keys | perm (Pcap + SPcap each)
    size_t bin_cap = 0;
    uint32_t* bin_hist = nullptr;    // histogram | offsets (BIN_MAX + 1 each)
    DevCtrl* ctrl = nullptr;
    uint32_t* h_active = nullptr;  // pinned ring of read-backs
    static constexpr int RING = 16;
    cudaEvent_t ring_ev[RING] = {};
    cudaEvent_t ev_begin = nullptr, ev_end = nullptr;
    std::vector<cudaEvent_t> ext_ev;  // per iteration: 4 events bracketing k_bin_* | k_traverse | k_shade
    unsigned char* d_rgb = nullptr;
    size_t rgb_cap = 0;
    unsigned char* h_rgb = nullptr;   // pinned
    size_t h_rgb_cap = 0;
    int32_t* d_probe = nullptr;
    size_t probe_cap = 0;
    volatile unsigned long long* h_state = nullptr;   // mapped pinned {iteration, live paths} (graph mode)
    unsigned long long* d_state = nullptr;
    cudaGraphExec_t graph_exec[4] = {nullptr, nullptr, nullptr, nullptr};   // one iteration (4 kernels) for cur = 0 / 1; [2], [3]: the same with the inline-tail k_shade ...
    std::vector<unsigned char> graph_args;                 // ... captured for exactly these kernel arguments
    int grid_shade_nomesh = 0;   // grid of the mesh-less k_shade instantiation (160-thread CTAs)
    int grid_shade_nee = 0;      // grid of the live-NEE mesh instantiations (SHADE_THREADS_NEE); grid_shade: the others
    int grid_oct = 0;    // k_traverse_octree's own persistent grid
    int grid_ext = 0, grid_ext_count = 0, grid_sh = 0, grid_sh_count = 0, grid_gen = 0, grid_shade = 0, grid_bin = 0;
    // adaptive sampling (ensure_adaptive): allocated by the first adaptive request only
    float2* ad_mom = nullptr;          // [pixel] (mean, M2)
    size_t ad_mom_cap = 0;
    int32_t* ad_list = nullptr;        // [tile] the active tiles, ascending
    uint32_t* ad_tile_ks = nullptr;    // [tile] samples per pixel so far
    float* ad_tile_err = nullptr;      // [tile] error estimate after the tile's latest pass
    int ad_tiles_cap = 0;
    volatile int* h_ad_count = nullptr;   // mapped pinned: active tiles after k_compact_tiles
    int* d_ad_count = nullptr;
    // denoiser (ensure_denoise): allocated by the first denoised request only
    float4* dn_guides = nullptr;       // [pixel] albedo | depth, then [pixel] normal | object id
    float4* dn_buf = nullptr;          // two ping-pong [pixel] illumination | variance buffers
    size_t dn_cap = 0;                 // pixels

    ~RenderContext() {
        cudaSetDevice(device);
        if (stream) cudaStreamSynchronize(stream);
        cudaFree(qbuf); cudaFree(sbuf); cudaFree(accum); cudaFree(ctrl); cudaFree(d_rgb); cudaFree(d_probe);
        cudaFree(bin_buf); cudaFree(bin_hist);
        cudaFree(ad_mom); cudaFree(ad_list); cudaFree(ad_tile_ks); cudaFree(ad_tile_err);
        cudaFree(dn_guides); cudaFree(dn_buf);
        if (h_ad_count) cudaFreeHost((void*)h_ad_count);
        if (h_active) cudaFreeHost(h_active);
        if (h_state) cudaFreeHost((void*)h_state);
        for (auto& e : graph_exec) if (e) cudaGraphExecDestroy(e);
        if (h_rgb) cudaFreeHost(h_rgb);
        for (auto& e : ring_ev) if (e) cudaEventDestroy(e);
        for (auto& e : ext_ev) cudaEventDestroy(e);
        if (ev_begin) cudaEventDestroy(ev_begin);
        if (ev_end) cudaEventDestroy(ev_end);
        if (stream) cudaStreamDestroy(stream);
        if (copy_stream) cudaStreamDestroy(copy_stream);
    }
};

}  // namespace

struct rtb_scene {
    HostScene hs;
    FlatScene fs;
    int device = 0;
    DevSceneHeader h_hdr{};
    // one pinned staging block: header | prims | materials | triangle vertices | tri_obj | light cdf
    unsigned char* h_stage = nullptr;
    unsigned char* d_stage = nullptr;
    size_t stage_bytes = 0;
    size_t off_prims = 0, off_mats = 0, off_verts = 0, off_triobj = 0, off_cdf = 0;
    float4* d_tri_orig = nullptr;
    LbvhResult bvh;
    DevScene view{};
    rtb_scene_info info{};
    std::mutex mu;
    std::vector<RenderContext*> pool;
    rtb_stats last_stats{};
    cudaStream_t stream = nullptr;
    // RTB_ACCEL_OCTREE_REFERENCE: the reference's octrees, built on first use
    bool octrees_built = false;
    float4* d_oct_nodes = nullptr;
    float4* d_oct_tris = nullptr;
    int32_t* d_oct_roots = nullptr;
    int oct_nodes = 0, oct_refs = 0;
    double oct_build_ms = 0;

    ~rtb_scene() {
        if (device < 0) return;
        cudaSetDevice(device);
        for (auto* c : pool) delete c;
        cudaFree(d_oct_nodes);
        cudaFree(d_oct_tris);
        cudaFree(d_oct_roots);
        free_lbvh(bvh);
        cudaFree(d_stage);
        cudaFree(d_tri_orig);
        if (h_stage) cudaFreeHost(h_stage);
        if (stream) cudaStreamDestroy(stream);
    }
};

namespace {

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

__global__ void k_tri_orig(const float* __restrict__ verts, int n, float4* __restrict__ out) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float* v = verts + (size_t)i * 9;
    out[3 * i] = make_float4(v[0], v[1], v[2], 0.f);
    out[3 * i + 1] = make_float4(v[3], v[4], v[5], 0.f);
    out[3 * i + 2] = make_float4(v[6], v[7], v[8], 0.f);
}

int upload_scene(rtb_scene* sc, uint64_t* bytes) {
    CU_TRY(cudaSetDevice(sc->device));
    CU_TRY(cudaMemcpyAsync(sc->d_stage, sc->h_stage, sc->stage_bytes, cudaMemcpyHostToDevice, sc->stream));
    CU_TRY(cudaStreamSynchronize(sc->stream));
    if (bytes) *bytes = sc->stage_bytes;
    return RTB_OK;
}

// LBVH tables of an exported scene (rtb_scene_export): host copies, laid out like the device arrays
struct LbvhImport {
    LbvhResult meta;   // scalars; the pointers are unused
    int n_tris;
    const float4 *nodes, *tris, *tri_nrm;
    const uint4* qnodes;
};

int build_device_scene(rtb_scene* sc, const LbvhImport* import = nullptr) {
    const FlatScene& fs = sc->fs;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(RTB_ECUDA, std::string("no CUDA device (librtb200 has no CPU fallback): ") + cudaGetErrorString(e));
    if (sc->device < 0 || sc->device >= ndev) return fail(RTB_EINVAL, "device ordinal out of range");
    CU_TRY(cudaSetDevice(sc->device));
    CU_TRY(cudaStreamCreateWithFlags(&sc->stream, cudaStreamNonBlocking));

    const int n_tris = (int)fs.tri_obj.size();
    sc->off_prims = align_up(sizeof(DevSceneHeader), 256);
    sc->off_mats = align_up(sc->off_prims + fs.prims.size() * sizeof(DevPrim), 256);
    sc->off_verts = align_up(sc->off_mats + fs.materials.size() * sizeof(DevMaterial), 256);
    sc->off_triobj = align_up(sc->off_verts + fs.tri_verts.size() * sizeof(float), 256);
    sc->off_cdf = align_up(sc->off_triobj + fs.tri_obj.size() * sizeof(int32_t), 256);
    // the light table of RTB_EST_NEE_ALL_LIGHTS (light_rule.cuh) goes behind the other tables; only the header knows where
    std::vector<DevLight> lights;
    std::vector<float> light_cdf;
    std::vector<int32_t> light_of((size_t)fs.n_objects, -1);
    {
        double cum = 0;
        for (size_t k = 0; k < fs.lights.size(); ++k) {
            cum += fs.lights[k].prob;
            light_cdf.push_back(k + 1 == fs.lights.size() ? 1.0f : (float)cum);
        }
        for (size_t k = 0; k < fs.lights.size(); ++k) {
            const FlatLight& l = fs.lights[k];
            const HostObject& o = sc->hs.objects[(size_t)l.obj];
            DevLight d{};
            d.sphere = make_float4((float)o.pos.x, (float)o.pos.y, (float)o.pos.z, (float)o.r);
            d.pdf_area = (float)(l.prob / l.area);
            d.obj = l.obj;
            d.tri_cdf = l.tri_cdf.empty() ? -1 : (int32_t)light_cdf.size();
            for (double c : l.tri_cdf) light_cdf.push_back((float)c);
            lights.push_back(d);
            light_of[(size_t)l.obj] = (int32_t)k;
        }
    }
    const size_t off_lights = align_up(sc->off_cdf + fs.light_cdf.size() * sizeof(float), 256);
    const size_t off_light_cdf = align_up(off_lights + lights.size() * sizeof(DevLight), 256);
    const size_t off_light_of = align_up(off_light_cdf + light_cdf.size() * sizeof(float), 256);
    sc->stage_bytes = align_up(off_light_of + light_of.size() * sizeof(int32_t), 256);
    CU_TRY(cudaMallocHost((void**)&sc->h_stage, sc->stage_bytes));
    CU_TRY(cudaMalloc((void**)&sc->d_stage, sc->stage_bytes));
    std::memset(sc->h_stage, 0, sc->stage_bytes);
    if (!lights.empty()) {
        std::memcpy(sc->h_stage + off_lights, lights.data(), lights.size() * sizeof(DevLight));
        std::memcpy(sc->h_stage + off_light_cdf, light_cdf.data(), light_cdf.size() * sizeof(float));
    }
    std::memcpy(sc->h_stage + off_light_of, light_of.data(), light_of.size() * sizeof(int32_t));
    if (!fs.prims.empty()) std::memcpy(sc->h_stage + sc->off_prims, fs.prims.data(), fs.prims.size() * sizeof(DevPrim));
    std::memcpy(sc->h_stage + sc->off_mats, fs.materials.data(), fs.materials.size() * sizeof(DevMaterial));
    if (n_tris) {
        std::memcpy(sc->h_stage + sc->off_verts, fs.tri_verts.data(), fs.tri_verts.size() * sizeof(float));
        std::memcpy(sc->h_stage + sc->off_triobj, fs.tri_obj.data(), fs.tri_obj.size() * sizeof(int32_t));
    }
    if (!fs.light_cdf.empty()) std::memcpy(sc->h_stage + sc->off_cdf, fs.light_cdf.data(), fs.light_cdf.size() * sizeof(float));

    // geometry first (the header needs the BVH root and box)
    CU_TRY(cudaMemcpyAsync(sc->d_stage, sc->h_stage, sc->stage_bytes, cudaMemcpyHostToDevice, sc->stream));
    const float* d_verts = reinterpret_cast<const float*>(sc->d_stage + sc->off_verts);
    const int32_t* d_triobj = reinterpret_cast<const int32_t*>(sc->d_stage + sc->off_triobj);
    cudaEvent_t e0, e1;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    CU_TRY(cudaEventRecord(e0, sc->stream));
    std::string err;
    if (import) {   // the tables another rank built: copy instead of building (the scene + BVH broadcast of a multi-GPU job)
        LbvhResult& B = sc->bvh;
        B = import->meta;
        B.d_nodes = nullptr; B.d_qnodes = nullptr; B.d_tris = nullptr; B.d_tri_nrm = nullptr;
        if (import->n_tris != n_tris) return fail(RTB_EPARSE, "exported scene: triangle count does not match the LBVH tables");
        auto up = [&](void** dst, const void* src, size_t bytes) -> cudaError_t {
            cudaError_t e = cudaMalloc(dst, std::max<size_t>(bytes, 16));
            if (e == cudaSuccess && bytes) e = cudaMemcpyAsync(*dst, src, bytes, cudaMemcpyHostToDevice, sc->stream);
            return e;
        };
        if (n_tris) {
            CU_TRY(up((void**)&B.d_nodes, import->nodes, (size_t)B.n_nodes * 4 * sizeof(float4)));
            CU_TRY(up((void**)&B.d_qnodes, import->qnodes, (size_t)B.n_nodes * 2 * sizeof(uint4)));
            CU_TRY(up((void**)&B.d_tris, import->tris, (size_t)n_tris * TRI_STRIDE * sizeof(float4)));
            CU_TRY(up((void**)&B.d_tri_nrm, import->tri_nrm, (size_t)n_tris * sizeof(float4)));
        }
    } else if (!build_lbvh(d_verts, d_triobj, n_tris, sc->stream, sc->bvh, err))
        return fail(err.rfind("unsupported:", 0) == 0 ? RTB_EUNSUPPORTED : RTB_ECUDA, err);
    if (n_tris) {
        CU_TRY(cudaMalloc((void**)&sc->d_tri_orig, (size_t)n_tris * 3 * sizeof(float4)));
        k_tri_orig<<<(n_tris + 255) / 256, 256, 0, sc->stream>>>(d_verts, n_tris, sc->d_tri_orig);
    }
    CU_TRY(cudaEventRecord(e1, sc->stream));
    CU_TRY(cudaStreamSynchronize(sc->stream));
    float build_ms = 0;
    CU_TRY(cudaEventElapsedTime(&build_ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);

    DevSceneHeader& H = sc->h_hdr;
    std::memset(&H, 0, sizeof(H));
    for (int k = 0; k < 3; ++k) {
        H.cam_pos[k] = fs.cam_pos[k];
        H.cam_dir[k] = fs.cam_dir[k];
        H.bvh_min[k] = sc->bvh.bmin[k];
        H.bvh_max[k] = sc->bvh.bmax[k];
    }
    H.n_prims = (int)fs.prims.size();
    H.n_objects = fs.n_objects;
    H.light_obj = fs.light_obj;
    H.light_geom = fs.light_geom;
    H.light_prim = -1;
    for (size_t k = 0; k < fs.prims.size(); ++k)
        if (fs.prims[k].obj == fs.light_obj) H.light_prim = (int)k;
    H.light_first_tri = fs.materials[fs.light_obj].first_tri;
    H.light_n_tri = fs.materials[fs.light_obj].n_tri;
    H.light_area = fs.light_area;
    H.n_tris = n_tris;
    H.root = sc->bvh.root;
    H.n_lights = (int32_t)lights.size();
    H.lights_select = lights.size() > 1 || (lights.size() == 1 && lights[0].tri_cdf >= 0);
    H.off_lights = (int32_t)(off_lights / 256);
    H.off_light_cdf = (int32_t)(off_light_cdf / 256);
    H.off_light_of = (int32_t)(off_light_of / 256);
    std::memcpy(sc->h_stage, &H, sizeof(H));
    CU_TRY(cudaMemcpyAsync(sc->d_stage, sc->h_stage, sizeof(H), cudaMemcpyHostToDevice, sc->stream));
    CU_TRY(cudaStreamSynchronize(sc->stream));

    DevScene& V = sc->view;
    V.hdr = reinterpret_cast<const DevSceneHeader*>(sc->d_stage);
    V.prims = reinterpret_cast<const DevPrim*>(sc->d_stage + sc->off_prims);
    V.mats = reinterpret_cast<const DevMaterial*>(sc->d_stage + sc->off_mats);
    V.qnodes = sc->bvh.d_qnodes;
    V.qmin = make_float3(sc->bvh.qmin[0], sc->bvh.qmin[1], sc->bvh.qmin[2]);
    V.qstep = make_float3(sc->bvh.qstep[0], sc->bvh.qstep[1], sc->bvh.qstep[2]);
    V.tris = sc->bvh.d_tris;
    V.tri_nrm = sc->bvh.d_tri_nrm;
    V.light_cdf = reinterpret_cast<const float*>(sc->d_stage + sc->off_cdf);
    V.tri_orig = sc->d_tri_orig;
    V.n_prims = H.n_prims;
    V.n_planes = fs.n_planes;
    V.n_objects = H.n_objects;
    V.n_tris = n_tris;
    V.root = H.root;
    V.bvh_min = make_float3(H.bvh_min[0], H.bvh_min[1], H.bvh_min[2]);
    V.bvh_max = make_float3(H.bvh_max[0], H.bvh_max[1], H.bvh_max[2]);

    rtb_scene_info& I = sc->info;
    std::memset(&I, 0, sizeof(I));
    I.n_objects = fs.n_objects;
    I.n_planes = fs.n_planes;
    I.n_spheres = fs.n_spheres;
    I.n_meshes = fs.n_meshes;
    I.n_triangles = n_tris;
    I.light_object = fs.light_obj;
    I.bvh_nodes = sc->bvh.n_nodes;
    I.bvh_leaves = sc->bvh.n_leaves;
    I.bvh_depth = sc->bvh.depth;
    I.device = sc->device;
    for (int k = 0; k < 3; ++k) {
        I.bvh_min[k] = H.bvh_min[k];
        I.bvh_max[k] = H.bvh_max[k];
        I.camera_pos[k] = fs.cam_pos[k];
        I.camera_dir[k] = fs.cam_dir[k];
    }
    I.build_ms = build_ms;
    return RTB_OK;
}

int finish_scene(rtb_scene* sc, int rc, const std::string& err, rtb_scene** out, const LbvhImport* import = nullptr) {
    if (rc != RTB_OK) {
        delete sc;
        return fail(rc, err);
    }
    std::string e2;
    rc = flatten_scene(sc->hs, sc->fs, e2);
    if (rc != RTB_OK) {
        delete sc;
        return fail(rc, e2);
    }
    if (sc->device < 0) {  // host-only handle (loader checks without a GPU): no device state at all
        rtb_scene_info& I = sc->info;
        std::memset(&I, 0, sizeof(I));
        I.n_objects = sc->fs.n_objects;
        I.n_planes = sc->fs.n_planes;
        I.n_spheres = sc->fs.n_spheres;
        I.n_meshes = sc->fs.n_meshes;
        I.n_triangles = (int)sc->fs.tri_obj.size();
        I.light_object = sc->fs.light_obj;
        I.device = -1;
        for (int k = 0; k < 3; ++k) { I.camera_pos[k] = sc->fs.cam_pos[k]; I.camera_dir[k] = sc->fs.cam_dir[k]; }
        *out = sc;
        return RTB_OK;
    }
    rc = build_device_scene(sc, import);
    if (rc != RTB_OK) {
        std::string keep = g_last_error;
        delete sc;
        g_last_error = keep;
        return rc;
    }
    *out = sc;
    return RTB_OK;
}

// ---------------------------------------------------------------- the reference's octrees (RTB_ACCEL_OCTREE_REFERENCE)
// Built on first use: Octree::build per mesh on the host in f64 (octree_host.cpp), flattened into one node table whose
// leaves reference the LBVH's triangle table (the LBVH build reordered the triangles: its `global id` column gives the
// inverse map), uploaded once.  Afterwards sc->view carries the tables and every render may ask for either accel mode.
int ensure_octrees(rtb_scene* sc) {
    std::lock_guard<std::mutex> lk(sc->mu);
    if (sc->octrees_built) return RTB_OK;
    CU_TRY(cudaSetDevice(sc->device));
    const auto t0 = std::chrono::steady_clock::now();
    const int n_tris = sc->view.n_tris;
    std::vector<int32_t> slot_of((size_t)n_tris, -1);   // global triangle index -> slot in the LBVH triangle table
    std::vector<float4> tris_host((size_t)n_tris * TRI_STRIDE);
    if (n_tris) {
        std::vector<float4>& tris = tris_host;
        CU_TRY(cudaMemcpy(tris.data(), sc->bvh.d_tris, tris.size() * sizeof(float4), cudaMemcpyDeviceToHost));
        for (int s = 0; s < n_tris; ++s) {
            int g;
            std::memcpy(&g, &tris[(size_t)s * TRI_STRIDE + 1].w, 4);
            if (g < 0 || g >= n_tris) return fail(RTB_ECUDA, "internal error: LBVH triangle table holds an invalid triangle id");
            slot_of[(size_t)g] = s;
        }
    }
    std::vector<float4> nodes;
    std::vector<int32_t> refs, roots;
    auto as_f = [](int v) { float f; std::memcpy(&f, &v, 4); return f; };
    for (int i = 0; i < sc->fs.n_objects; ++i) {
        const HostObject& ob = sc->hs.objects[(size_t)i];
        if (ob.geom != GEOM_MESH) continue;
        HostOctree ot;
        build_reference_octree(ob, ot);
        if (ot.nodes.empty()) { roots.push_back(-1); continue; }
        const int node_base = (int)(nodes.size() / 2), ref_base = (int)refs.size();
        const int first_tri = sc->fs.materials[(size_t)i].first_tri;
        roots.push_back(node_base);
        // breadth-first renumbering: the children of a parent become neighbours, in octant order (octree.cuh: node record)
        std::vector<int> bfs{0}, first_child(ot.nodes.size(), 0);
        for (size_t q = 0; q < bfs.size(); ++q) {
            const HostOctreeNode& n = ot.nodes[(size_t)bfs[q]];
            if (n.count >= 0) continue;
            first_child[(size_t)bfs[q]] = (int)bfs.size();
            for (int k = 0; k < 8; ++k) if (n.child[k] >= 0) bfs.push_back(n.child[k]);
        }
        for (int old_index : bfs) {
            const HostOctreeNode& n = ot.nodes[(size_t)old_index];
            int mask = 0;
            for (int k = 0; k < 8; ++k) if (n.child[k] >= 0) mask |= 1 << k;
            const bool leaf = n.count >= 0;
            nodes.push_back(make_float4((float)n.mn[0], (float)n.mn[1], (float)n.mn[2], as_f(leaf ? ref_base + n.first : node_base + first_child[(size_t)old_index])));
            nodes.push_back(make_float4((float)n.mx[0], (float)n.mx[1], (float)n.mx[2], as_f(leaf ? n.count : -1 - mask)));
        }
        for (int32_t t : ot.tri_refs) refs.push_back(slot_of[(size_t)(first_tri + t)]);
    }
    if (!nodes.empty()) {
        CU_TRY(cudaMalloc((void**)&sc->d_oct_nodes, nodes.size() * sizeof(float4)));
        CU_TRY(cudaMemcpy(sc->d_oct_nodes, nodes.data(), nodes.size() * sizeof(float4), cudaMemcpyHostToDevice));
    }
    if (!refs.empty()) {   // every reference gets its own copy of the triangle record; [1].w (the global triangle id there) names the slot in the LBVH table
        std::vector<float4> rt(refs.size() * TRI_STRIDE);
        for (size_t k = 0; k < refs.size(); ++k) {
            for (int q = 0; q < TRI_STRIDE; ++q) rt[k * TRI_STRIDE + q] = tris_host[(size_t)refs[k] * TRI_STRIDE + q];
            rt[k * TRI_STRIDE + 1].w = as_f(refs[k]);
        }
        CU_TRY(cudaMalloc((void**)&sc->d_oct_tris, rt.size() * sizeof(float4)));
        CU_TRY(cudaMemcpy(sc->d_oct_tris, rt.data(), rt.size() * sizeof(float4), cudaMemcpyHostToDevice));
    }
    if (!roots.empty()) {
        CU_TRY(cudaMalloc((void**)&sc->d_oct_roots, roots.size() * sizeof(int32_t)));
        CU_TRY(cudaMemcpy(sc->d_oct_roots, roots.data(), roots.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    }
    sc->view.oct_nodes = sc->d_oct_nodes;
    sc->view.oct_tris = sc->d_oct_tris;
    sc->view.oct_roots = sc->d_oct_roots;
    sc->view.n_oct_meshes = (int)roots.size();
    sc->oct_nodes = (int)(nodes.size() / 2);
    sc->oct_refs = (int)refs.size();
    sc->oct_build_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    sc->info.octree_nodes = sc->oct_nodes;
    sc->info.octree_tri_refs = sc->oct_refs;
    sc->octrees_built = true;
    return RTB_OK;
}

// ---------------------------------------------------------------- render contexts
// want_paths: path slots the caller is going to ask for — the pooled context whose queues fit best is handed out
// (smallest that is large enough, else the largest), so that nothing is reallocated when it can be avoided
RenderContext* acquire_context(rtb_scene* sc, uint32_t want_paths = 0) {
    std::lock_guard<std::mutex> lk(sc->mu);
    if (!sc->pool.empty()) {
        size_t best = 0;
        for (size_t k = 1; k < sc->pool.size(); ++k) {
            const uint32_t a = sc->pool[k]->Palloc, b = sc->pool[best]->Palloc;
            const bool a_fits = a >= want_paths, b_fits = b >= want_paths;
            if ((a_fits && (!b_fits || a < b)) || (!a_fits && !b_fits && a > b)) best = k;
        }
        RenderContext* c = sc->pool[best];
        sc->pool.erase(sc->pool.begin() + (long)best);
        return c;
    }
    RenderContext* c = new RenderContext();
    c->device = sc->device;
    return c;
}
void release_context(rtb_scene* sc, RenderContext* c) {
    if (!c->initialised) {   // ensure_context failed half-way: do not hand a half-built context to the next render
        delete c;
        return;
    }
    std::lock_guard<std::mutex> lk(sc->mu);
    sc->pool.push_back(c);
}

int default_bin_bits();
// the FIRST octree kernel ran one ray per thread through a deeply branching search (5.8 of 32 lanes active): there neighbouring
// lanes that walk neighbouring octants in the same order did pay (bench frame at 64 spp: traversal 800 -> 638 ms with 4 cell
// bits per axis, 601 with 5, for 73 / 125 ms of binning: frame 892 -> 803 ms).  The persistent, stepwise kernel that replaced it
// does not need the help: 496 ms unbinned, 554 ms with 4 bits.  Off by default; rtb_params.tuning[3] still selects it.
#ifndef RTB_OCTREE_BIN_BITS
#define RTB_OCTREE_BIN_BITS 0
#endif
constexpr int OCTREE_BIN_BITS = RTB_OCTREE_BIN_BITS;
// cell bits per axis of the coherence binning this request asks for (0 = off):
// rtb_params.tuning[3] & 255 = 0 library default | 1 off | 2..5 bits
int requested_bin_bits(const rtb_scene* sc, const rtb_params* p) {
    if (sc->view.n_tris == 0) return 0;   // scenes without triangles never traverse
    const int code = p->tuning[3] & 255;
    const int dflt = p->accel == RTB_ACCEL_OCTREE_REFERENCE ? OCTREE_BIN_BITS : default_bin_bits();
    return code == 0 ? dflt : (code == 1 ? 0 : std::min(std::max(code, 2), BIN_MAX_BITS));
}

int ensure_context(rtb_scene* sc, RenderContext* c, uint32_t P, uint32_t SP, size_t accum_elems, bool binning = false) {
    CU_TRY(cudaSetDevice(sc->device));
    if (!c->initialised) {   // a context whose set-up failed half-way is deleted by its caller, never pooled
        CU_TRY(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        CU_TRY(cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
        CU_TRY(cudaMalloc((void**)&c->ctrl, sizeof(DevCtrl)));
        CU_TRY(cudaMallocHost((void**)&c->h_active, sizeof(uint32_t) * RenderContext::RING));
        CU_TRY(cudaHostAlloc((void**)&c->h_state, 2 * sizeof(unsigned long long), cudaHostAllocMapped));
        CU_TRY(cudaHostGetDevicePointer((void**)&c->d_state, (void*)c->h_state, 0));
        for (auto& e : c->ring_ev) CU_TRY(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CU_TRY(cudaEventCreate(&c->ev_begin));
        CU_TRY(cudaEventCreate(&c->ev_end));
        const size_t smem_tab = shared_tables_bytes(sc->view.n_prims, sc->view.n_objects);
        const size_t smem_stack = shared_stack_bytes(WF_THREADS);
        cudaDeviceProp prop;
        CU_TRY(cudaGetDeviceProperties(&prop, sc->device));
        // The attribute is per kernel, not per scene: always opt in to the largest table set
        // (MAX_OBJECTS primitives + materials), never to this scene's own (smaller) size.
        const int smem_max = (int)shared_tables_bytes(MAX_OBJECTS, MAX_OBJECTS);
        CU_TRY(cudaFuncSetAttribute(k_shade<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        CU_TRY(cudaFuncSetAttribute(k_shade<1, 0, 0, true, SHADE_THREADS_NEE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        CU_TRY(cudaFuncSetAttribute(k_shade<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        CU_TRY(cudaFuncSetAttribute(k_shade<3>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        CU_TRY(cudaFuncSetAttribute(k_shade<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        CU_TRY(cudaFuncSetAttribute(k_shade<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        CU_TRY(cudaFuncSetAttribute(k_generate<0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
        const int smem_tail = (int)shared_scene_bytes(MAX_OBJECTS, MAX_OBJECTS, SHADE_THREADS);
        const int smem_tail_nee = (int)shared_scene_bytes(MAX_OBJECTS, MAX_OBJECTS, SHADE_THREADS_NEE);
        CU_TRY(cudaFuncSetAttribute(k_shade<0, 0, 0, true, SHADE_THREADS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_tail));
        CU_TRY(cudaFuncSetAttribute(k_shade<1, 0, 0, true, SHADE_THREADS_NEE, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_tail_nee));
        CU_TRY(cudaFuncSetAttribute(k_shade<2, 0, 0, true, SHADE_THREADS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_tail));
        CU_TRY(cudaFuncSetAttribute(k_shade<3, 0, 0, true, SHADE_THREADS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_tail));
        CU_TRY(cudaFuncSetAttribute(k_shade<4, 0, 0, true, SHADE_THREADS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_tail));
        CU_TRY(cudaFuncSetAttribute(k_shade<5, 0, 0, true, SHADE_THREADS, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_tail));
        int b = 0;
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, k_traverse<false>, WF_THREADS, smem_stack));
        c->grid_ext = std::max(1, b) * prop.multiProcessorCount;
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, k_traverse<true>, WF_THREADS, smem_stack));
        c->grid_ext_count = std::max(1, b) * prop.multiProcessorCount;
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, k_traverse_octree<false>, WF_THREADS, (size_t)OCT_MAX_DEPTH * WF_THREADS * sizeof(int2)));
        c->grid_oct = std::max(1, b) * prop.multiProcessorCount;
        // the queued k_shade instantiations of one CTA shape share a grid: it is sized for the one with the fewest CTAs per SM
        // (their register counts differ; the inline-tail instantiations, limited by their stacks, may run in more than one wave)
        auto shade_grid = [&](std::initializer_list<const void*> kernels, int threads, int& grid) -> int {
            int fewest = INT_MAX;
            for (const void* k : kernels) {
                CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, k, threads, smem_tab));
                fewest = std::min(fewest, b);
            }
            grid = std::max(1, fewest) * prop.multiProcessorCount;
            return RTB_OK;
        };
        if (int e = shade_grid({(const void*)k_shade<0>, (const void*)k_shade<2>, (const void*)k_shade<2, 8, 0>, (const void*)k_shade<2, 5, 1>,
                                (const void*)k_shade<2, 5, 2>, (const void*)k_shade<2, 5, 3>, (const void*)k_shade<3>, (const void*)k_shade<4>,
                                (const void*)k_shade<5>}, SHADE_THREADS, c->grid_shade)) return e;
        if (int e = shade_grid({(const void*)k_shade<1, 0, 0, true, SHADE_THREADS_NEE>, (const void*)k_shade<1, 8, 0, true, SHADE_THREADS_NEE>,
                                (const void*)k_shade<1, 5, 1, true, SHADE_THREADS_NEE>, (const void*)k_shade<1, 5, 2, true, SHADE_THREADS_NEE>,
                                (const void*)k_shade<1, 5, 3, true, SHADE_THREADS_NEE>}, SHADE_THREADS_NEE, c->grid_shade_nee)) return e;
        if (int e = shade_grid({(const void*)k_shade<1, 5, 3, false, SHADE_THREADS_NOMESH>, (const void*)k_shade<2, 5, 3, false, SHADE_THREADS_NOMESH>},
                               SHADE_THREADS_NOMESH, c->grid_shade_nomesh)) return e;
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, k_generate<0, 0>, WF_THREADS, smem_tab));
        c->grid_gen = std::max(1, b) * prop.multiProcessorCount;
        c->grid_bin = 8 * prop.multiProcessorCount;
        // experiment knobs: CTAs per SM of the two persistent kernels (two concurrent renders can then share every SM)
        if (const char* e = getenv("RTB_TRAV_CTAS")) c->grid_ext = c->grid_ext_count = std::max(1, atoi(e)) * prop.multiProcessorCount;
        if (const char* e = getenv("RTB_SHADE_CTAS")) c->grid_shade = c->grid_shade_nee = std::max(1, atoi(e)) * prop.multiProcessorCount;
        c->initialised = true;
    }
    // every k_shade warp may leave up to two unfilled SHADE_SEG segments per queue class behind in each iteration
    const uint32_t seg_room = (uint32_t)std::max({c->grid_shade * (SHADE_THREADS / 32), c->grid_shade_nee * (SHADE_THREADS_NEE / 32),
                                                  c->grid_shade_nomesh * (SHADE_THREADS_NOMESH / 32)}) * 2u * SHADE_SEG;
    {
        const uint32_t cap = P + 2u * seg_room;   // front + back class
        if (c->Palloc < cap) {   // (re)allocation of GBs of queue costs 100s of ms: never shrink, so a scene that serves
            cudaFree(c->qbuf);   // whole frames and band-sized streaming jobs alternately does it once
            c->qbuf = nullptr;
            c->Palloc = 0;
            CU_TRY(cudaMalloc((void**)&c->qbuf, (size_t)cap * 9 * sizeof(float4)));
            c->Palloc = cap;
        }
        c->P = P;
        c->Pcap = cap;
    }
    {
        // 2 x SP: a path that queued a shadow ray may stay in registers (k_shade, `sh_tight`) while the shadow queue holds fewer than SP
        // entries; from then on it is parked as before, which adds at most one entry (two under the dead-MIS estimator: SP is 2 P
        // there) per path and iteration
        const uint32_t cap = 2u * SP + seg_room;
        if (c->SPalloc < cap) {
            cudaFree(c->sbuf);
            c->sbuf = nullptr;
            c->SPalloc = 0;
            CU_TRY(cudaMalloc((void**)&c->sbuf, (size_t)cap * 6 * sizeof(float4)));
            c->SPalloc = cap;
        }
        c->SP = SP;
        c->SPcap = cap;
    }
    if (c->accum_cap < accum_elems) {
        cudaFree(c->accum);
        c->accum = nullptr;
        CU_TRY(cudaMalloc((void**)&c->accum, accum_elems * sizeof(float4)));
        c->accum_cap = accum_elems;
    }
    if (binning) {   // coherence binning of the LBVH rays: buffers exist only once a request asks for it
        const size_t need = (size_t)c->Pcap + c->SPcap;
        if (c->bin_cap < need) {
            cudaFree(c->bin_buf);
            c->bin_buf = nullptr;
            c->bin_cap = 0;
            CU_TRY(cudaMalloc((void**)&c->bin_buf, need * 2 * sizeof(uint32_t)));
            c->bin_cap = need;
        }
        if (!c->bin_hist) {
            CU_TRY(cudaMalloc((void**)&c->bin_hist, (size_t)(BIN_MAX + 1) * 2 * sizeof(uint32_t)));
            CU_TRY(cudaMemsetAsync(c->bin_hist, 0, (size_t)(BIN_MAX + 1) * 2 * sizeof(uint32_t), c->stream));
        }
    }
    return RTB_OK;
}

int ensure_octrees(rtb_scene* sc);
// the tables the requested accel mode needs exist (the reference's octrees are built on first use)
int need_accel(rtb_scene* sc, const rtb_params* p) {
    if (p->accel == RTB_ACCEL_OCTREE_REFERENCE && sc->view.n_tris > 0) return ensure_octrees(sc);
    return RTB_OK;
}

int need_device(const rtb_scene* sc) {
    if (!sc) return fail(RTB_EINVAL, "NULL scene");
    if (sc->device < 0) return fail(RTB_ECUDA, "host-only scene handle (device = -1): no CUDA device owns it, and there is no CPU fallback");
    return RTB_OK;
}

int check_params(const rtb_params* p) {
    if (!p) return fail(RTB_EINVAL, "params is NULL");
    if (p->width <= 0 || p->height <= 0 || p->width > 65535 || p->height > 65535)
        return fail(RTB_EINVAL, "width/height must be in 1..65535 (the wire format carries u16 coordinates)");
    if (p->spp < 0) return fail(RTB_EINVAL, "spp must be >= 0");
    if ((long long)p->spp / 4 * 4 >= (1 << 20)) return fail(RTB_EINVAL, "spp too large (sample index field is 20 bits)");
    if (p->world < 1 || p->rank < 0 || p->rank >= p->world) return fail(RTB_EINVAL, "need 0 <= rank < world");
    if (p->estimator != RTB_EST_NEE && p->estimator != RTB_EST_MIS_DEAD && p->estimator != RTB_EST_MIS_BALANCE && p->estimator != RTB_EST_NEE_ALL_LIGHTS)
        return fail(RTB_EINVAL, "unknown estimator");
    if ((long long)p->width * p->height * 4 >= (1ll << 31)) return fail(RTB_EINVAL, "frame too large for 31-bit accumulator indices");
    if (p->accel != RTB_ACCEL_LBVH && p->accel != RTB_ACCEL_OCTREE_REFERENCE) return fail(RTB_EINVAL, "unknown accel mode");
    return RTB_OK;
}

// shadow-queue slots for P paths: the NEE estimators queue at most one shadow ray per vertex, the MIS ones two
uint32_t shadow_slots(int estimator, uint32_t P) {
    return estimator == RTB_EST_NEE || estimator == RTB_EST_NEE_ALL_LIGHTS ? P : 2 * P;
}

int local_tiles(const rtb_params* p) {
    int tx = (p->width + TILE - 1) / TILE, ty = (p->height + TILE - 1) / TILE;
    int T = tx * ty;
    return T > p->rank ? (T - p->rank + p->world - 1) / p->world : 0;
}

// Path slots in flight.  More slots = fewer, fuller wavefront iterations (measured on flying_unicorn 1080p 256 spp:
// 8 Mi 497, 16 Mi 528, 32 Mi 542 Msamples/s), but 240 B of queue memory each; default: one eighth of the frame's
// samples, between 1 Mi and 32 Mi (7.7 GB); tools/gpu_pool_small.py has the small-frame sweep.
uint32_t pool_for(uint64_t samples, int pool_paths) {
    uint64_t P;
    if (pool_paths > 0) P = (uint64_t)pool_paths;
    else {
        // one eighth of the work keeps the regeneration tail short; a frame of at most 2 Mi samples goes through in ONE wave
        uint64_t want = std::max<uint64_t>(samples / 8, std::min<uint64_t>(samples, 2ull << 20));
        P = 1ull << 20;
        while (P < want && P < (1ull << 25)) P <<= 1;
    }
    P = std::max<uint64_t>(P, 1024);
    return (uint32_t)((P + 31ull) & ~31ull);
}
uint32_t default_pool(const rtb_params* p) {
    return pool_for((uint64_t)local_tiles(p) * 1024ull * 4ull * (uint64_t)std::max(1, p->spp / 4), p->pool_paths);
}

// library default of the coherence binning (cell bits per axis, 0 = off); RTB_BIN_BITS overrides it
int default_bin_bits() {
    static const int v = [] {
        const char* e = getenv("RTB_BIN_BITS");
        return e ? std::min(std::max(atoi(e), 0), BIN_MAX_BITS) : 0;
    }();
    return v;
}

// every mesh query of one iteration: the LBVH kernel (the product's fast path) or the reference's octrees
void launch_traverse(RenderContext* c, const RenderArgs& a, int cur, bool count_work, size_t smem_stack) {
    if (a.accel == RTB_ACCEL_OCTREE_REFERENCE) {
        // persistent like k_traverse (its own grid, the same work cursor); shared memory = the per-thread stack of parent nodes
        const size_t smem_oct = (size_t)OCT_MAX_DEPTH * WF_THREADS * sizeof(int2);
        if (count_work) k_traverse_octree<true><<<c->grid_oct, WF_THREADS, smem_oct, c->stream>>>(a, cur);
        else k_traverse_octree<false><<<c->grid_oct, WF_THREADS, smem_oct, c->stream>>>(a, cur);
    } else if (count_work) k_traverse<true><<<c->grid_ext_count, WF_THREADS, smem_stack, c->stream>>>(a, cur);
    else k_traverse<false><<<c->grid_ext, WF_THREADS, smem_stack, c->stream>>>(a, cur);
}

void launch_binning(RenderContext* c, const RenderArgs& a, int cur) {
    if (a.bin_bits <= 0) return;
    k_bin_keys<<<c->grid_bin, WF_THREADS, 0, c->stream>>>(a, cur);
    k_bin_scan<<<1, BIN_SCAN_THREADS, 0, c->stream>>>(a);
    k_bin_scatter<<<c->grid_bin, WF_THREADS, 0, c->stream>>>(a, cur);
}

void fill_args(const rtb_scene* sc, const rtb_params* p, RenderContext* c, RenderArgs& a) {
    std::memset(&a, 0, sizeof(a));
    {   // (callers asking for RTB_ACCEL_OCTREE_REFERENCE have run ensure_octrees first: need_accel; another thread may be inside it now)
        std::lock_guard<std::mutex> lk(const_cast<rtb_scene*>(sc)->mu);
        a.S = sc->view;
    }
    a.cam = make_camera(sc->fs.cam_pos, sc->fs.cam_dir, p->width, p->height);
    a.width = p->width;
    a.height = p->height;
    a.spp = p->spp;
    a.num_samples = p->spp / 4;
    a.ks_done = (uint32_t)(p->spp / 4) * 4u;
    a.keys = philox_keys((uint32_t)p->seed, (uint32_t)(p->seed >> 32));
    a.estimator = p->estimator;
    a.tune_refill = p->tuning[1];
    a.tune_steps = p->tuning[2];
    a.accel = p->accel;
    a.rank = p->rank;
    a.world = p->world;
    a.tiles_x = (p->width + TILE - 1) / TILE;
    a.tiles_y = (p->height + TILE - 1) / TILE;
    a.n_local_tiles = local_tiles(p);
    a.P = c->P;
    a.SP = c->SP;
    a.Pcap = c->Pcap;
    a.SPcap = c->SPcap;
    for (int k = 0; k < 2; ++k) {
        float4* b = c->qbuf + (size_t)k * 4 * c->Pcap;
        a.q[k].o = b;
        a.q[k].d = b + c->Pcap;
        a.q[k].beta = b + 2 * (size_t)c->Pcap;
        a.q[k].ov = b + 3 * (size_t)c->Pcap;
        a.q[k].hit = reinterpret_cast<float2*>(c->qbuf + (size_t)8 * c->Pcap) + (size_t)k * c->Pcap;
    }
    for (int k = 0; k < 2; ++k) {
        float4* b = c->sbuf + (size_t)k * 3 * c->SPcap;
        a.sq[k].o = b;
        a.sq[k].d = b + c->SPcap;
        a.sq[k].c = b + 2 * (size_t)c->SPcap;
    }
    a.accum = c->accum;
    a.ctrl = c->ctrl;
    for (const FlatPrim& P : sc->fs.prims)
        if (P.obj == sc->fs.light_obj && sc->fs.light_geom == GEOM_SPHERE) {
            a.light_sphere = make_float4(P.a[0], P.a[1], P.a[2], P.a[3]);
            a.light_pdf = 1.0f / (4.0f * 3.14159265358979323846f * P.a[3] * P.a[3]);
        }
    if (sc->fs.prims.size() <= 8)
        for (size_t k = 0; k < sc->fs.prims.size(); ++k) {
            const FlatPrim& P = sc->fs.prims[k];
            a.ss.a[k] = make_float4(P.a[0], P.a[1], P.a[2], P.a[3]);
            a.ss.r2[k] = P.b[0];
            a.ss.group[k] = P.group;
        }
    a.trav_warps = (uint32_t)c->grid_ext * (WF_THREADS / 32);
    a.shade_warps = (uint32_t)c->grid_shade * (SHADE_THREADS / 32);
    // coherence binning: rtb_params.tuning[3] = 0 library default | 1 off | 2..5 cell bits per axis, + 256 = octant-major keys
    a.bin_bits = c->bin_buf && c->bin_hist ? requested_bin_bits(sc, p) : 0;
    a.bin_octant_major = (p->tuning[3] >> 8) & 1;
    a.bin_key = c->bin_buf;
    a.bin_perm = c->bin_buf ? c->bin_buf + c->bin_cap : nullptr;
    a.bin_hist = c->bin_hist;
    a.bin_offs = c->bin_hist ? c->bin_hist + (BIN_MAX + 1) : nullptr;
}

static RenderArgs with_cur(const RenderArgs& a, int cur) {
    RenderArgs r = a;
    r.qin = a.q[cur];
    r.qout = a.q[1 - cur];
    r.sqin = a.sq[cur];
    r.sqout = a.sq[1 - cur];
    return r;
}
static void launch_generate(int n_planes, int n_spheres, int grid, size_t smem, cudaStream_t st, const RenderArgs& a, int cur) {
    const bool small = n_planes == 5 && n_spheres >= 1 && n_spheres <= 3 && !getenv("RTB_NO_SMALL_TABLE");
    if (!small) k_generate<0, 0><<<grid, WF_THREADS, smem, st>>>(a, cur);
    else if (n_spheres == 1) k_generate<5, 1><<<grid, WF_THREADS, smem, st>>>(a, cur);
    else if (n_spheres == 2) k_generate<5, 2><<<grid, WF_THREADS, smem, st>>>(a, cur);
    else k_generate<5, 3><<<grid, WF_THREADS, smem, st>>>(a, cur);
}
// k_shade instantiations: general | reference-scene fast paths | fast paths with the analytic table in the kernel
// parameters, unrolled for 5 planes + 1..3 spheres (cubes, flying_unicorn, cornell_box)
static bool shade_is_nomesh(int mode, const RenderArgs& a) {
    return a.S.n_tris == 0 && (mode == 1 || mode == 2) && a.S.n_planes == 5 && a.S.n_prims - a.S.n_planes == 3 && !getenv("RTB_NO_SMALL_TABLE") &&
           !getenv("RTB_GENERIC_TABLE");
}
// paths left below which a run switches to the inline-tail k_shade (0 = never); RTB_INLINE_TAIL overrides
uint32_t inline_tail_below() {   // read per run: tests and A/B tools flip it inside one process
    const char* e = getenv("RTB_INLINE_TAIL");
    return e ? (uint32_t)std::max(0, atoi(e)) : (2u << 20);   // measured: gains saturate between 1 Mi and 4 Mi paths
}

// The CTA shape follows the mode (shade_cta): `grid` must be the grid of that shape, as a.shade_warps counts its warps.
static void launch_shade(int mode, int n_planes, int n_spheres, int grid, size_t smem, cudaStream_t st, const RenderArgs& a, int cur, bool inline_tail = false) {
#define RTB_SHADE(M, P, S) k_shade<M, P, S, true, shade_cta(M)><<<grid, shade_cta(M), smem, st>>>(a, cur)
    if (inline_tail) {   // the tail of a run: k_shade traverses the LBVH itself (generic analytic table; + the traversal stack in shared memory)
        const size_t smem_t = shared_scene_bytes(a.S.n_prims, a.S.n_objects, shade_cta(mode));
        if (mode == 1) k_shade<1, 0, 0, true, shade_cta(1), true><<<grid, shade_cta(1), smem_t, st>>>(a, cur);
        else if (mode == 2) k_shade<2, 0, 0, true, shade_cta(2), true><<<grid, shade_cta(2), smem_t, st>>>(a, cur);
        else if (mode == 3) k_shade<3, 0, 0, true, shade_cta(3), true><<<grid, shade_cta(3), smem_t, st>>>(a, cur);
        else if (mode == 4) k_shade<4, 0, 0, true, shade_cta(4), true><<<grid, shade_cta(4), smem_t, st>>>(a, cur);
        else if (mode == 5) k_shade<5, 0, 0, true, shade_cta(5), true><<<grid, shade_cta(5), smem_t, st>>>(a, cur);
        else k_shade<0, 0, 0, true, shade_cta(0), true><<<grid, shade_cta(0), smem_t, st>>>(a, cur);
        return;
    }
    if (shade_is_nomesh(mode, a)) {
        // cornell_box: analytic primitives only
        if (mode == 1) k_shade<1, 5, 3, false, SHADE_THREADS_NOMESH><<<grid, SHADE_THREADS_NOMESH, smem, st>>>(a, cur);
        else k_shade<2, 5, 3, false, SHADE_THREADS_NOMESH><<<grid, SHADE_THREADS_NOMESH, smem, st>>>(a, cur);
        return;
    }
    const bool small = mode != 0 && n_planes == 5 && n_spheres >= 1 && n_spheres <= 3 && !getenv("RTB_NO_SMALL_TABLE") && !getenv("RTB_GENERIC_TABLE");
    if (mode == 1 && small) { if (n_spheres == 1) RTB_SHADE(1, 5, 1); else if (n_spheres == 2) RTB_SHADE(1, 5, 2); else RTB_SHADE(1, 5, 3); }
    else if (mode == 2 && small) { if (n_spheres == 1) RTB_SHADE(2, 5, 1); else if (n_spheres == 2) RTB_SHADE(2, 5, 2); else RTB_SHADE(2, 5, 3); }
    else if (mode == 1 && n_planes + n_spheres <= 8 && !getenv("RTB_NO_SMALL_TABLE")) RTB_SHADE(1, 8, 0);   // any small scene: generic unrolled table
    else if (mode == 2 && n_planes + n_spheres <= 8 && !getenv("RTB_NO_SMALL_TABLE")) RTB_SHADE(2, 8, 0);
    else if (mode == 1) RTB_SHADE(1, 0, 0);
    else if (mode == 2) RTB_SHADE(2, 0, 0);
    else if (mode == 3) RTB_SHADE(3, 0, 0);
    else if (mode == 4) RTB_SHADE(4, 0, 0);
    else if (mode == 5) RTB_SHADE(5, 0, 0);
    else RTB_SHADE(0, 0, 0);
#undef RTB_SHADE
}

// The wavefront loop: runs samples [ks_begin, ks_end) (ks = k*4 + sub-pixel) of every local pixel,
// or the n_probe explicit items.  Accumulators are NOT cleared here.
int run_wavefront(rtb_scene* sc, RenderContext* c, RenderArgs& a, uint32_t ks_begin, uint32_t ks_end, bool count_work,
                  volatile int* cancel, rtb_stats& st, bool& cancelled) {
    cancelled = false;
    a.trav_warps = (uint32_t)(a.accel == RTB_ACCEL_OCTREE_REFERENCE ? c->grid_oct : (count_work ? c->grid_ext_count : c->grid_ext)) * (WF_THREADS / 32);   // must match the launched grid
    a.shade_warps = (uint32_t)c->grid_shade * (SHADE_THREADS / 32);
    DevCtrl h{};
    h.ext_head(0) = h.ext_head(1) = 0;
    h.ext_tail(0) = h.ext_tail(1) = a.Pcap;
    h.sh_head(0) = h.sh_head(1) = 0;
    unsigned long long npl = a.pixel_list ? (unsigned long long)a.n_probe : (unsigned long long)a.n_local_tiles * 1024ull;
    const bool explicit_items = a.probe_px && !a.pixel_list;
    h.work_next = explicit_items ? 0ull : (unsigned long long)ks_begin * npl;
    h.work_total = explicit_items ? (unsigned long long)a.n_probe : (unsigned long long)ks_end * npl;
    h.tile_base = a.tile_base;
    h.n_tiles = a.n_local_tiles;
    CU_TRY(cudaMemcpyAsync(c->ctrl, &h, sizeof(h), cudaMemcpyHostToDevice, c->stream));
    CU_TRY(cudaEventRecord(c->ev_begin, c->stream));
    const size_t smem_tab = shared_tables_bytes(a.S.n_prims, a.S.n_objects);
    const size_t smem_stack = shared_stack_bytes(WF_THREADS);
    uint64_t launches = 0;
    size_t ext_iters = 0;
    int cur = 0;
    uint64_t it = 0;
    bool done = h.work_total == h.work_next;
    // Small frames are launch-bound (four tiny kernels per iteration): replay one captured CUDA graph per
    // iteration and let k_prepare publish the live-path count to mapped host memory instead of copying it back.
    // compile-time specialisation of k_shade for the common case (see its definition)
    if (a.estimator == RTB_EST_MIS_BALANCE && sc->fs.light_geom != GEOM_SPHERE)
        return fail(RTB_EUNSUPPORTED, "RTB_EST_MIS_BALANCE needs a sphere light (the reference's mesh-light sampler does not return points of the mesh, src/geometry.rs:622-628)");
    // a scene with a dielectric always runs the general kernel with the dielectric branch (MODE 3), probes included
    bool dielectric = false;
    for (const FlatMaterial& m : sc->fs.materials) dielectric = dielectric || m.brdf == BRDF_DIELECTRIC;
    bool fast_shade = !a.probe_px && a.estimator != RTB_EST_MIS_BALANCE && sc->fs.light_geom == GEOM_SPHERE && !getenv("RTB_NO_FAST_SHADE");
    for (const FlatMaterial& m : sc->fs.materials) fast_shade = fast_shade && m.brdf != BRDF_PHONG;
    // RTB_EST_NEE_ALL_LIGHTS: the general kernel with next-event estimation over the whole light table (MODE 4), or MODE 3's
    // dielectric kernel with it (MODE 5), probes included
    const int shade_mode = a.estimator == RTB_EST_NEE_ALL_LIGHTS ? (dielectric ? 5 : 4)
                                                                 : (dielectric ? 3 : (!fast_shade ? 0 : (a.estimator == 0 ? 1 : 2)));
    // the CTA shape of k_shade depends on the instantiation: so do its grid and warp count (static first chunks, k_prepare)
    const bool nomesh = shade_is_nomesh(shade_mode, a);
    const int grid_shade = nomesh ? c->grid_shade_nomesh : (shade_mode == 1 ? c->grid_shade_nee : c->grid_shade);
    a.shade_warps = (uint32_t)grid_shade * (uint32_t)(shade_cta(shade_mode, !nomesh) / 32);
    // the inline tail: once at most `tail_below` paths are left, k_shade traverses the LBVH itself and the run ends in one launch
    // (the LBVH only: the reference's octree search and the counting build keep the queued form)
    // — and never more than a quarter of the pool: a run whose pool is that small would otherwise spend its WHOLE life in the
    // inline form, which costs 3-4 x per path (measured: 600x450x64 with a 1 Mi pool, 97 vs 26 ms)
    const uint32_t tail_below = (a.S.n_tris > 0 && !nomesh && !count_work && a.accel == RTB_ACCEL_LBVH) ? std::min(inline_tail_below(), a.P / 4u) : 0u;
    bool tail_mode = false;
    uint32_t graph_max_pool = 1u << 24;
    if (const char* e = getenv("RTB_GRAPH_MAX_POOL")) graph_max_pool = (uint32_t)std::max(0, atoi(e));   // experiment knob
    const bool use_graph = !count_work && a.P <= graph_max_pool && !getenv("RTB_NO_GRAPH");
    if (use_graph && !done) {
        RenderArgs ag = a;
        ag.host_state = c->d_state;
        ag.tile_base = ag.n_local_tiles = 0;   // the kernels of the loop read the tile range from the control block: one graph serves every band
        c->h_state[0] = 0;
        c->h_state[1] = 1;
        cudaError_t ge = cudaSuccess;
        const bool cached = c->graph_exec[0] && (!tail_below || c->graph_exec[2]) && c->graph_args.size() == sizeof(RenderArgs) &&
                            std::memcmp(c->graph_args.data(), &ag, sizeof(RenderArgs)) == 0;
        if (!cached) {   // progressive passes re-use the graphs: the sample range lives in the control block, not in the arguments
            for (auto& e : c->graph_exec) if (e) { cudaGraphExecDestroy(e); e = nullptr; }
            for (int k = 0; k < (tail_below ? 4 : 2) && ge == cudaSuccess; ++k) {   // [0], [1]: the queued form; [2], [3]: the inline tail
                cudaGraph_t g = nullptr;
                ge = cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal);
                if (ge != cudaSuccess) break;
                const int par = k & 1;
                k_prepare<<<1, 1, 0, c->stream>>>(ag, par);
                const RenderArgs agk = with_cur(ag, par);   // queue pointers of this parity, resolved here
                launch_generate(a.S.n_planes, a.S.n_prims - a.S.n_planes, c->grid_gen, smem_tab, c->stream, agk, par);
                launch_binning(c, agk, par);
                launch_traverse(c, agk, par, false, smem_stack);
                launch_shade(shade_mode, a.S.n_planes, a.S.n_prims - a.S.n_planes, grid_shade, smem_tab, c->stream, agk, par, k >= 2);
                ge = cudaStreamEndCapture(c->stream, &g);
                if (ge == cudaSuccess) ge = cudaGraphInstantiate(&c->graph_exec[k], g, 0);
                if (g) cudaGraphDestroy(g);
            }
            if (ge != cudaSuccess) {
                for (auto& e : c->graph_exec) if (e) { cudaGraphExecDestroy(e); e = nullptr; }
                c->graph_args.clear();
                return fail(RTB_ECUDA, std::string("graph capture: ") + cudaGetErrorString(ge));
            }
            c->graph_args.assign(reinterpret_cast<unsigned char*>(&ag), reinterpret_cast<unsigned char*>(&ag) + sizeof(RenderArgs));
        }
        cudaGraphExec_t* exec = c->graph_exec;
        // graphs launched beyond the newest iteration the device has reported: enough to hide the launch latency of the
        // short tail iterations, few enough that a finished run leaves only a handful of empty graphs behind (each costs
        // ~8 us of device time — most of a 1-sample progressive pass when there were 24 of them)
        const uint64_t run_ahead = 6;
        while (!done) {
            if (cancel && *cancel) { cancelled = true; break; }
            ge = cudaGraphLaunch(exec[cur + (tail_mode ? 2 : 0)], c->stream);
            if (ge != cudaSuccess) break;
            launches += a.bin_bits > 0 ? 7 : 4;
            ++it;
            cur ^= 1;
            for (;;) {   // {iteration, live paths} as published by the newest k_prepare that has run
                const unsigned long long seen = c->h_state[0];
                if (tail_below && seen >= 1 && c->h_state[1] <= tail_below && c->h_state[0] == seen) tail_mode = true;
                if (seen >= 1 && c->h_state[1] == 0 && c->h_state[0] == seen) { done = true; break; }
                if (it - seen < run_ahead) break;
                if (cudaStreamQuery(c->stream) == cudaSuccess && c->h_state[0] == seen && it - seen >= run_ahead) {
                    // everything launched has run; the published state is final for those iterations
                    if (c->h_state[1] == 0) done = true;
                    break;
                }
            }
        }
        cudaError_t se = cudaStreamSynchronize(c->stream);
        if (ge != cudaSuccess || se != cudaSuccess) {
            cudaGetLastError();   // do not leave the error for the next call to trip over
            return fail(RTB_ECUDA, std::string("graph launch: ") + cudaGetErrorString(ge != cudaSuccess ? ge : se));
        }
        done = true;
    }
    int outstanding = 0;
    uint64_t oldest = 0;
    while (!done) {
        if (cancel && *cancel) { cancelled = true; break; }
        k_prepare<<<1, 1, 0, c->stream>>>(a, cur);
        const RenderArgs ac = with_cur(a, cur);
        launch_generate(a.S.n_planes, a.S.n_prims - a.S.n_planes, c->grid_gen, smem_tab, c->stream, ac, cur);
        while (c->ext_ev.size() < 4 * (ext_iters + 1)) {
            cudaEvent_t e0;
            CU_TRY(cudaEventCreate(&e0));
            c->ext_ev.push_back(e0);
        }
        cudaEvent_t* ev = &c->ext_ev[4 * ext_iters];
        CU_TRY(cudaEventRecord(ev[3], c->stream));
        launch_binning(c, ac, cur);
        CU_TRY(cudaEventRecord(ev[0], c->stream));
        launch_traverse(c, ac, cur, count_work, smem_stack);
        CU_TRY(cudaEventRecord(ev[1], c->stream));
        launch_shade(shade_mode, a.S.n_planes, a.S.n_prims - a.S.n_planes, grid_shade, smem_tab, c->stream, ac, cur, tail_mode);
        CU_TRY(cudaEventRecord(ev[2], c->stream));
        ++ext_iters;
        launches += a.bin_bits > 0 ? 7 : 4;
        // lagged, non-blocking termination test: read back `active` (state after this iteration's
        // k_prepare) into a pinned ring; the host keeps launching until a completed read-back says 0.
        int slot = (int)(it % RenderContext::RING);
        CU_TRY(cudaMemcpyAsync(&c->h_active[slot], &c->ctrl->active, sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
        CU_TRY(cudaEventRecord(c->ring_ev[slot], c->stream));
        ++outstanding;
        ++it;
        cur ^= 1;
        while (outstanding > 0) {
            int s = (int)(oldest % RenderContext::RING);
            // at most 6 iterations ahead of the newest count the host has seen (like the graph path): the switch to the inline tail and
            // the end of the run are noticed that much sooner (bench frame: 82 -> 6x iterations)
            cudaError_t q = outstanding >= 6 ? cudaEventSynchronize(c->ring_ev[s]) : cudaEventQuery(c->ring_ev[s]);
            if (q == cudaErrorNotReady) break;
            if (q != cudaSuccess) return fail(RTB_ECUDA, std::string("wavefront loop: ") + cudaGetErrorString(q));
            if (c->h_active[s] == 0) done = true;
            else if (tail_below && c->h_active[s] <= tail_below) tail_mode = true;
            ++oldest;
            --outstanding;
        }
    }
    CU_TRY(cudaEventRecord(c->ev_end, c->stream));
    CU_TRY(cudaMemcpyAsync(&h, c->ctrl, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    CU_TRY(cudaGetLastError());
    float ms = 0;
    CU_TRY(cudaEventElapsedTime(&ms, c->ev_begin, c->ev_end));
    double ext_ms = 0, shade_ms = 0, shadow_ms = 0;   // shadow_ms: the binning kernels (rtb_stats.bin_ms)
    for (size_t k = 0; k < ext_iters; ++k) {
        float m = 0;
        CU_TRY(cudaEventElapsedTime(&m, c->ext_ev[4 * k], c->ext_ev[4 * k + 1]));
        ext_ms += m;
        CU_TRY(cudaEventElapsedTime(&m, c->ext_ev[4 * k + 1], c->ext_ev[4 * k + 2]));
        shade_ms += m;
        CU_TRY(cudaEventElapsedTime(&m, c->ext_ev[4 * k + 3], c->ext_ev[4 * k]));
        shadow_ms += m;
    }
    if (h.overflow) return fail(RTB_ECUDA, "internal error: " + std::to_string(h.overflow) + " queue slots beyond the physical capacity were refused (frame is incomplete)");
    st.samples += h.samples;
    st.rays_primary += h.rays_primary;
    st.rays_extension += h.rays_extension;
    st.rays_shadow += h.rays_shadow;
    st.iterations += h.iterations;
    st.kernel_launches += launches;
    st.bvh_node_visits += h.node_visits;
    st.bvh_tri_tests += h.tri_tests;
    if (count_work && getenv("RTB_DEBUG_TRAVERSE"))
        fprintf(stderr, "[rtb] traverse slots: rounds %llu inner-offered %llu used %llu (%.1f%%) | leaf phases %llu lanes %llu (%.1f of 32) | refills %llu lanes %llu (%.1f per refill)\n",
                h.dbg[0], h.dbg[1], h.node_visits, 100.0 * h.node_visits / (double)std::max<unsigned long long>(1, h.dbg[1]), h.dbg[2], h.dbg[3],
                (double)h.dbg[3] / (double)std::max<unsigned long long>(1, h.dbg[2]), h.dbg[4], h.dbg[5], (double)h.dbg[5] / (double)std::max<unsigned long long>(1, h.dbg[4]));
    st.render_ms += ms;
    st.extend_ms += ext_ms;
    st.shade_ms += shade_ms;
    st.bin_ms += shadow_ms;
    st.rays_bvh += h.rays_bvh;
    st.shadow_bvh += h.shadow_bvh;
    st.paths_queued += h.paths_queued;
    return RTB_OK;
}

// full render of this rank's tiles into the context's accumulators, then resolve
int render_into_context(rtb_scene* sc, const rtb_params* p, RenderContext* c, RenderArgs& a, volatile int* cancel, rtb_stats& st,
                        bool& cancelled) {
    uint32_t P = default_pool(p);
    uint32_t SP = shadow_slots(p->estimator, P);
    size_t accum_elems = (size_t)p->width * p->height * 4;
    int rc = ensure_context(sc, c, P, SP, accum_elems, requested_bin_bits(sc, p) > 0);
    if (rc != RTB_OK) return rc;
    fill_args(sc, p, c, a);
    CU_TRY(cudaMemsetAsync(c->accum, 0, accum_elems * sizeof(float4), c->stream));
    st = rtb_stats{};
    cancelled = false;
    if (a.num_samples > 0 && a.n_local_tiles > 0) {
        bool count_work = p->tuning[0] == 1;
        rc = run_wavefront(sc, c, a, 0u, (uint32_t)a.num_samples * 4u, count_work, cancel, st, cancelled);
        if (rc != RTB_OK) return rc;
    }
    return RTB_OK;
}

int resolve_to(RenderContext* c, const RenderArgs& a, unsigned char* d_out, float4* d_sub, int scanline, rtb_stats& st) {
    int n = a.n_local_tiles * 1024;
    if (n == 0) return RTB_OK;
    cudaEvent_t e0 = c->ev_begin, e1 = c->ev_end;
    CU_TRY(cudaEventRecord(e0, c->stream));
    k_resolve<<<(n + 255) / 256, 256, 0, c->stream>>>(a, d_out, d_sub, scanline);
    CU_TRY(cudaEventRecord(e1, c->stream));
    CU_TRY(cudaStreamSynchronize(c->stream));
    CU_TRY(cudaGetLastError());
    float ms = 0;
    CU_TRY(cudaEventElapsedTime(&ms, e0, e1));
    st.resolve_ms += ms;
    st.kernel_launches += 1;
    return RTB_OK;
}

void publish_stats(rtb_scene* sc, const rtb_stats& st, bool calling_thread = true) {
    if (calling_thread) {
        g_thread_stats = st;
        g_thread_stats_scene = sc;
    }
    std::lock_guard<std::mutex> lk(sc->mu);
    sc->last_stats = st;
}

int ensure_rgb(RenderContext* c, size_t bytes, bool host) {
    if (c->rgb_cap < bytes) {
        cudaFree(c->d_rgb);
        c->d_rgb = nullptr;
        CU_TRY(cudaMalloc((void**)&c->d_rgb, bytes));
        c->rgb_cap = bytes;
    }
    if (host && c->h_rgb_cap < bytes) {
        if (c->h_rgb) cudaFreeHost(c->h_rgb);
        c->h_rgb = nullptr;
        CU_TRY(cudaMallocHost((void**)&c->h_rgb, bytes));
        c->h_rgb_cap = bytes;
    }
    return RTB_OK;
}

// ---------------------------------------------------------------- adaptive sampling
// host-side checks only (a host-only scene reaches them): the error names the offending field
int check_adaptive(const rtb_params* p, const rtb_adaptive* o) {
    if (!o) return fail(RTB_EINVAL, "rtb_adaptive options are NULL");
    if (!std::isfinite(o->target_levels) || o->target_levels < 0.f) return fail(RTB_EINVAL, "rtb_adaptive.target_levels must be finite and >= 0");
    if (o->pass_spp <= 0 || o->pass_spp % 4 != 0) return fail(RTB_EINVAL, "rtb_adaptive.pass_spp must be a positive multiple of 4");
    if (p->spp % o->pass_spp != 0) return fail(RTB_EINVAL, "params.spp (the budget) must be a multiple of rtb_adaptive.pass_spp");
    if (o->min_spp % o->pass_spp != 0 || o->min_spp < 2 * o->pass_spp || o->min_spp > p->spp)
        return fail(RTB_EINVAL, "rtb_adaptive.min_spp must be a multiple of pass_spp in [2 * pass_spp, spp]");
    if (o->reserved != 0) return fail(RTB_EINVAL, "rtb_adaptive.reserved must be 0");
    if (p->world != 1) return fail(RTB_EINVAL, "adaptive rendering renders whole frames (params.world must be 1)");
    return RTB_OK;
}

// path slots of one pass over the whole frame (later passes hold fewer tiles)
uint32_t adaptive_pool(const rtb_params* p, const rtb_adaptive* o) {
    return pool_for((uint64_t)local_tiles(p) * 1024ull * (uint64_t)o->pass_spp, p->pool_paths);
}

int ensure_adaptive(RenderContext* c, int n_tiles, size_t pixels) {
    if (!c->h_ad_count) {
        CU_TRY(cudaHostAlloc((void**)&c->h_ad_count, sizeof(int), cudaHostAllocMapped));
        CU_TRY(cudaHostGetDevicePointer((void**)&c->d_ad_count, (void*)c->h_ad_count, 0));
    }
    if (c->ad_mom_cap < pixels) {
        cudaFree(c->ad_mom);
        c->ad_mom = nullptr;
        c->ad_mom_cap = 0;
        CU_TRY(cudaMalloc((void**)&c->ad_mom, pixels * sizeof(float2)));
        c->ad_mom_cap = pixels;
    }
    if (c->ad_tiles_cap < n_tiles) {
        cudaFree(c->ad_list); cudaFree(c->ad_tile_ks); cudaFree(c->ad_tile_err);
        c->ad_list = nullptr; c->ad_tile_ks = nullptr; c->ad_tile_err = nullptr;
        c->ad_tiles_cap = 0;
        CU_TRY(cudaMalloc((void**)&c->ad_list, (size_t)n_tiles * sizeof(int32_t)));
        CU_TRY(cudaMalloc((void**)&c->ad_tile_ks, (size_t)n_tiles * sizeof(uint32_t)));
        CU_TRY(cudaMalloc((void**)&c->ad_tile_err, (size_t)n_tiles * sizeof(float)));
        c->ad_tiles_cap = n_tiles;
    }
    return RTB_OK;
}

void add_stats(rtb_stats& d, const rtb_stats& s);

// The adaptive pass loop (world = 1): clears the accumulators, then renders pass after pass — samples
// [pass * pass_spp, (pass + 1) * pass_spp) of the budget frame's numbering, so a tile's samples are a prefix of the budget
// frame's — over the tiles still in the list, until none is left.  `after_pass` (may be empty) runs once per pass with that
// pass's counters, once k_adapt has advanced tile_ks.  On return a.tile_ks holds the per-tile sample counts for k_resolve.
int run_adaptive(rtb_scene* sc, RenderContext* c, RenderArgs& a, const rtb_adaptive& o, volatile int* cancel, rtb_stats& st,
                 bool& cancelled, const std::function<int(int, const rtb_stats&)>& after_pass) {
    const int n_tiles = a.tiles_x * a.tiles_y;
    const size_t pixels = (size_t)a.width * a.height;
    int rc = ensure_adaptive(c, n_tiles, pixels);
    if (rc != RTB_OK) return rc;
    AdaptArgs ad{c->accum, c->ad_mom, c->ad_list, c->ad_tile_ks, c->ad_tile_err, a.width, a.height, a.tiles_x,
                 o.pass_spp, a.spp, o.min_spp, o.target_levels};
    CU_TRY(cudaMemsetAsync(c->accum, 0, pixels * 4 * sizeof(float4), c->stream));
    CU_TRY(cudaMemsetAsync(c->ad_mom, 0, pixels * sizeof(float2), c->stream));
    k_adapt_init<<<(n_tiles + 255) / 256, 256, 0, c->stream>>>(ad, n_tiles);
    st.kernel_launches += 1;
    RenderArgs r = a;   // the list pointer stays the same from pass to pass: run_wavefront's captured graphs are re-used
    r.tile_base = 0;
    r.tile_list = c->ad_list;
    cancelled = false;
    for (int pass = 0, count = n_tiles; count > 0; ++pass) {
        const uint32_t k0 = (uint32_t)pass * (uint32_t)o.pass_spp;
        r.n_local_tiles = count;
        rtb_stats ps{};
        rc = run_wavefront(sc, c, r, k0, k0 + (uint32_t)o.pass_spp, false, cancel, ps, cancelled);
        if (rc != RTB_OK || cancelled) return rc;
        k_adapt<<<count, ADAPT_THREADS, 0, c->stream>>>(ad);
        k_compact_tiles<<<1, COMPACT_THREADS, 0, c->stream>>>(c->ad_list, count, c->d_ad_count);
        CU_TRY(cudaStreamSynchronize(c->stream));
        CU_TRY(cudaGetLastError());
        count = *c->h_ad_count;
        ps.kernel_launches += 2;
        add_stats(st, ps);
        if (after_pass && (rc = after_pass(pass, ps)) != RTB_OK) return rc;
    }
    a.tile_ks = c->ad_tile_ks;
    return RTB_OK;
}

// ---------------------------------------------------------------- denoiser
// host-side checks only (a host-only scene reaches them): the error names the offending field; p = nullptr for
// rtb_denoise_image (no frame request)
int check_denoise(const rtb_params* p, const rtb_denoise* o) {
    if (!o) return fail(RTB_EINVAL, "rtb_denoise options are NULL");
    if (o->levels < 0 || o->levels > DENOISE_MAX_LEVELS) return fail(RTB_EINVAL, "rtb_denoise.levels must be in 0..8");
    if (!std::isfinite(o->sigma_color) || o->sigma_color < 0.f) return fail(RTB_EINVAL, "rtb_denoise.sigma_color must be finite and >= 0");
    if (!std::isfinite(o->sigma_normal) || o->sigma_normal < 0.f) return fail(RTB_EINVAL, "rtb_denoise.sigma_normal must be finite and >= 0");
    if (!std::isfinite(o->sigma_depth) || o->sigma_depth < 0.f) return fail(RTB_EINVAL, "rtb_denoise.sigma_depth must be finite and >= 0");
    for (int r : o->reserved)
        if (r != 0) return fail(RTB_EINVAL, "rtb_denoise.reserved must be 0");
    if (p && p->world != 1) return fail(RTB_EINVAL, "denoising filters whole frames (params.world must be 1)");
    return RTB_OK;
}

int ensure_denoise(RenderContext* c, size_t pixels) {
    if (c->dn_cap < pixels) {
        cudaFree(c->dn_guides); cudaFree(c->dn_buf);
        c->dn_guides = nullptr; c->dn_buf = nullptr;
        c->dn_cap = 0;
        CU_TRY(cudaMalloc((void**)&c->dn_guides, pixels * 2 * sizeof(float4)));
        CU_TRY(cudaMalloc((void**)&c->dn_buf, pixels * 2 * sizeof(float4)));
        c->dn_cap = pixels;
    }
    return RTB_OK;
}

// the guides of a width x height frame into c->dn_guides, enqueued on `st` (callers asking for RTB_ACCEL_OCTREE_REFERENCE have
// run need_accel)
int launch_gbuffer(rtb_scene* sc, RenderContext* c, int width, int height, int accel, cudaStream_t st) {
    DevScene S;
    {
        std::lock_guard<std::mutex> lk(sc->mu);
        S = sc->view;
    }
    const size_t pixels = (size_t)width * height;
    CU_TRY(cudaFuncSetAttribute(k_gbuffer, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shared_scene_bytes(MAX_OBJECTS, MAX_OBJECTS, WF_THREADS)));
    const Camera cam = make_camera(sc->fs.cam_pos, sc->fs.cam_dir, width, height);
    const int grid = (int)std::min<size_t>((pixels + WF_THREADS - 1) / WF_THREADS, 148 * 8);
    k_gbuffer<<<grid, WF_THREADS, shared_scene_bytes(S.n_prims, S.n_objects, WF_THREADS), st>>>(S, cam, width, height, accel, c->dn_guides,
                                                                                              c->dn_guides + pixels);
    CU_TRY(cudaGetLastError());
    return RTB_OK;
}

DenoiseArgs denoise_args(RenderContext* c, int width, int height) {
    DenoiseArgs d{};
    const size_t pixels = (size_t)width * height;
    d.width = width;
    d.height = height;
    d.tiles_x = (width + TILE - 1) / TILE;
    d.ga = c->dn_guides;
    d.gn = c->dn_guides + pixels;
    d.buf[0] = c->dn_buf;
    d.buf[1] = c->dn_buf + pixels;
    return d;
}

// the filter over d's buffers, enqueued on `st`: prep, o.levels à-trous levels, output; returns the kernels launched
int launch_filter(const DenoiseArgs& d, const rtb_denoise& o, unsigned char* rgb8, float* out3, cudaStream_t st) {
    const int n = d.width * d.height, grid = (n + DENOISE_THREADS - 1) / DENOISE_THREADS;
    const DenoiseSigmas s{o.sigma_color, o.sigma_normal, o.sigma_depth};
    k_denoise_prep<<<grid, DENOISE_THREADS, 0, st>>>(d);
    for (int level = 0; level < o.levels; ++level)
        k_atrous<<<grid, DENOISE_THREADS, 0, st>>>(d, d.buf[level & 1], d.buf[(level + 1) & 1], 1 << level, s);
    k_denoise_out<<<grid, DENOISE_THREADS, 0, st>>>(d, d.buf[o.levels & 1], rgb8, out3);
    return o.levels + 2;
}

// the denoised frame of the accumulators r describes (sample counts as r.ks_done / r.tile_ks give them) into rgb8 (scan-line);
// the guides must already be in c->dn_guides
int launch_denoise(RenderContext* c, const RenderArgs& r, const rtb_denoise& o, unsigned char* rgb8, cudaStream_t st) {
    DenoiseArgs d = denoise_args(c, r.width, r.height);
    d.accum = r.accum;
    d.ks_done = r.ks_done;
    d.tile_ks = r.tile_ks;
    return launch_filter(d, o, rgb8, nullptr, st);
}

// Whole-frame render (world = 1) of rtb_render_adaptive and rtb_render_denoised: the adaptive passes (opts) or one uniform
// pass, then k_resolve (dn = nullptr) or the denoiser, read back into rgb8_out.  Options are checked by the caller.
int render_whole_frame(rtb_scene* scene, const rtb_params* params, const rtb_adaptive* opts, const rtb_denoise* dn, uint8_t* rgb8_out,
                       int32_t* tile_spp, float* tile_error, volatile int* cancel) {
    int rc = need_device(scene);
    if (rc != RTB_OK) return rc;
    if ((rc = need_accel(scene, params)) != RTB_OK) return rc;
    const uint32_t P = opts ? adaptive_pool(params, opts) : default_pool(params);
    const uint32_t SP = shadow_slots(params->estimator, P);
    const size_t frame = (size_t)params->width * params->height * 3;
    const int n_tiles = local_tiles(params);
    RenderContext* c = acquire_context(scene, P);
    RenderArgs a;
    rtb_stats st{};
    bool cancelled = false;
    if (opts) {
        rc = ensure_context(scene, c, P, SP, (size_t)params->width * params->height * 4, requested_bin_bits(scene, params) > 0);
        if (rc == RTB_OK) {
            fill_args(scene, params, c, a);
            rc = run_adaptive(scene, c, a, *opts, cancel, st, cancelled, {});
        }
    } else {
        rc = render_into_context(scene, params, c, a, cancel, st, cancelled);
    }
    if (rc == RTB_OK && !cancelled) rc = ensure_rgb(c, frame, true);
    if (rc == RTB_OK && !cancelled) {
        if (!dn) rc = resolve_to(c, a, c->d_rgb, nullptr, 1, st);
        else if ((rc = ensure_denoise(c, (size_t)params->width * params->height)) == RTB_OK &&
                 (rc = launch_gbuffer(scene, c, params->width, params->height, params->accel, c->stream)) == RTB_OK) {
            cudaEvent_t e0 = c->ev_begin, e1 = c->ev_end;
            cudaError_t e = cudaEventRecord(e0, c->stream);
            if (e == cudaSuccess) st.kernel_launches += 1 + launch_denoise(c, a, *dn, c->d_rgb, c->stream);
            if (e == cudaSuccess) e = cudaEventRecord(e1, c->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
            if (e == cudaSuccess) e = cudaGetLastError();
            float ms = 0;
            if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, e0, e1);
            if (e != cudaSuccess) rc = fail(RTB_ECUDA, std::string("denoiser: ") + cudaGetErrorString(e));
            st.resolve_ms += ms;
        }
    }
    if (rc == RTB_OK && !cancelled) {
        cudaError_t e = cudaMemcpyAsync(c->h_rgb, c->d_rgb, frame, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess && opts && tile_spp) e = cudaMemcpyAsync(tile_spp, c->ad_tile_ks, (size_t)n_tiles * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess && opts && tile_error) e = cudaMemcpyAsync(tile_error, c->ad_tile_err, (size_t)n_tiles * sizeof(float), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) rc = fail(RTB_ECUDA, std::string("frame read-back: ") + cudaGetErrorString(e));
        else std::memcpy(rgb8_out, c->h_rgb, frame);
    }
    publish_stats(scene, st);
    release_context(scene, c);
    if (rc != RTB_OK) return rc;
    return cancelled ? RTB_ECANCELLED : RTB_OK;
}

}  // namespace

// ======================================================================================= C ABI
extern "C" {

const char* rtb_last_error(void) { return g_last_error.c_str(); }

int rtb_scene_load_toml(const char* toml_path, const char* assets_dir, int device, rtb_scene** out) {
    if (!toml_path || !out) return fail(RTB_EINVAL, "NULL argument");
    *out = nullptr;
    rtb_scene* sc = new rtb_scene();
    sc->device = device;
    std::string err;
    int rc = load_scene_file(toml_path, assets_dir ? assets_dir : "", sc->hs, err);
    return finish_scene(sc, rc, err, out);
}

int rtb_scene_load_toml_string(const char* toml_text, const char* assets_dir, int device, rtb_scene** out) {
    if (!toml_text || !out) return fail(RTB_EINVAL, "NULL argument");
    *out = nullptr;
    rtb_scene* sc = new rtb_scene();
    sc->device = device;
    std::string err;
    int rc = load_scene_text(toml_text, assets_dir ? assets_dir : "", sc->hs, err);
    return finish_scene(sc, rc, err, out);
}

int rtb_scene_create(const rtb_scene_desc* desc, int device, rtb_scene** out) {
    if (!desc || !out || (desc->n_objects > 0 && !desc->objects)) return fail(RTB_EINVAL, "NULL argument");
    *out = nullptr;
    rtb_scene* sc = new rtb_scene();
    sc->device = device;
    sc->hs.cam_pos = {desc->camera_pos[0], desc->camera_pos[1], desc->camera_pos[2]};
    sc->hs.cam_dir = {desc->camera_dir[0], desc->camera_dir[1], desc->camera_dir[2]};
    std::string err;
    int rc = RTB_OK;
    for (int i = 0; i < desc->n_objects && rc == RTB_OK; ++i) {
        const rtb_object_desc& d = desc->objects[i];
        HostObject o;
        o.emitted = {d.emitted[0], d.emitted[1], d.emitted[2]};
        if (d.brdf < 0 || d.brdf > 3 || d.geometry < 0 || d.geometry > 2) { rc = RTB_EPARSE; err = "object " + std::to_string(i) + ": unknown brdf / geometry kind"; break; }
        o.brdf = d.brdf;
        if (d.brdf == BRDF_PHONG) {
            if (d.k[2] < 0) { rc = RTB_EPARSE; err = "phong power must be >= 0"; break; }
            o.phong_kd = d.k[0]; o.phong_ks = d.k[1]; o.phong_power = (int)d.k[2];
            o.color_d = {d.color_d[0], d.color_d[1], d.color_d[2]};
            o.color_s = {d.color_s[0], d.color_s[1], d.color_s[2]};
        } else if (d.brdf == BRDF_DIELECTRIC) {
            if (!std::isfinite(d.k[0]) || !(d.k[0] > 0)) { rc = RTB_EPARSE; err = "object " + std::to_string(i) + ": dielectric ior (k[0]) must be a finite number > 0"; break; }
            bool tint_ok = true;
            for (int c = 0; c < 3; ++c) tint_ok = tint_ok && d.color_d[c] >= 0 && d.color_d[c] <= 1;
            if (!tint_ok) { rc = RTB_EPARSE; err = "object " + std::to_string(i) + ": dielectric tint (color_d) components must lie in [0, 1]"; break; }
            o.k = {d.k[0], 0, 0};
            o.color_d = {d.color_d[0], d.color_d[1], d.color_d[2]};
        } else {
            o.k = {d.k[0], d.k[1], d.k[2]};
        }
        o.geom = d.geometry;
        o.pos = {d.pos[0], d.pos[1], d.pos[2]};
        o.n = {d.n[0], d.n[1], d.n[2]};
        o.r = d.r;
        if (d.geometry == GEOM_MESH) {
            if (d.n_triangles <= 0 || !d.triangles) { rc = RTB_EMESH; err = "object " + std::to_string(i) + ": mesh has no faces"; break; }
            o.vertices.reserve((size_t)d.n_triangles * 3);
            for (int64_t t = 0; t < d.n_triangles * 3; ++t) {
                o.vertices.push_back({d.triangles[3 * t], d.triangles[3 * t + 1], d.triangles[3 * t + 2]});
                o.indices.push_back((uint32_t)t);
            }
            init_mesh_tables(o);
        }
        sc->hs.objects.push_back(std::move(o));
    }
    if (rc == RTB_OK) rc = finish_host_scene(sc->hs, err);
    return finish_scene(sc, rc, err, out);
}

// ---- scene + BVH as one blob: what a multi-GPU job broadcasts once (BASELINE.json north_star) --------------------
// Layout: ExportHeader | per object: ExportObject, vertices (3 f64 each), indices (u32), cumulative areas (f64) | LBVH tables
// (fp32 nodes, quantised nodes, triangles, normals) exactly as they sit in device memory.  A rank that imports the blob
// neither parses TOML / OBJ nor builds a BVH; it gets bit-identical tables, hence bit-identical traversal.
namespace {
struct ExportHeader {
    char magic[8];
    uint64_t total_bytes;
    double cam_pos[3], cam_dir[3];
    int32_t n_objects, light;
    int32_t n_tris, n_nodes, n_leaves, root, depth, pad[3];   // pad: zero; no implicit padding, build_ms stays at byte 152
    float qmin[3], qstep[3], bmin[3], bmax[3];
    double build_ms;
};
// build_ms is the one header field that differs between two builds of one scene: readers that compare blobs mask it
// at this offset
static_assert(offsetof(ExportHeader, build_ms) == 152, "ExportHeader layout changed: bump EXPORT_MAGIC");
struct ExportObject {
    double emitted[3], k[3], color_d[3], color_s[3], pos[3], n[3], bb_min[3], bb_max[3];
    double phong_kd, phong_ks, r, surface_area;
    int32_t brdf, phong_power, geom, pad;
    uint64_t n_vertices, n_indices, n_cum;
};
constexpr char EXPORT_MAGIC[8] = {'R', 'T', 'B', 'S', 'C', 'N', '3', 0};
void put3(double* d, const D3& v) { d[0] = v.x; d[1] = v.y; d[2] = v.z; }
D3 get3(const double* d) { return D3{d[0], d[1], d[2]}; }
size_t lbvh_bytes(const LbvhResult& B, int n_tris) {
    if (n_tris == 0) return 0;
    return (size_t)B.n_nodes * 4 * sizeof(float4) + (size_t)B.n_nodes * 2 * sizeof(uint4) + (size_t)n_tris * TRI_STRIDE * sizeof(float4) +
           (size_t)n_tris * sizeof(float4);
}
}  // namespace

int64_t rtb_scene_export(rtb_scene* scene, void* buf, int64_t cap) {
    if (!scene) return fail(RTB_EINVAL, "NULL scene");
    // a host-only handle (device = -1) exports the objects alone (n_tris = -1 in the header): the importer builds the LBVH itself
    const bool tables = scene->device >= 0;
    const int n_tris = tables ? scene->view.n_tris : 0;
    size_t total = sizeof(ExportHeader);
    for (const HostObject& o : scene->hs.objects)
        total += sizeof(ExportObject) + o.vertices.size() * 3 * sizeof(double) + o.indices.size() * sizeof(uint32_t) + o.cumulative_area.size() * sizeof(double);
    total = align_up(total, 16);
    const size_t lbvh_off = total;
    total += lbvh_bytes(scene->bvh, n_tris);
    if (!buf || cap < (int64_t)total) return (int64_t)total;   // size query
    unsigned char* p = static_cast<unsigned char*>(buf);
    ExportHeader H{};
    std::memcpy(H.magic, EXPORT_MAGIC, 8);
    H.total_bytes = total;
    put3(H.cam_pos, scene->hs.cam_pos);
    put3(H.cam_dir, scene->hs.cam_dir);
    H.n_objects = (int32_t)scene->hs.objects.size();
    H.light = scene->hs.light;
    const LbvhResult& B = scene->bvh;
    H.n_tris = tables ? n_tris : -1; H.n_nodes = B.n_nodes; H.n_leaves = B.n_leaves; H.root = B.root; H.depth = B.depth;
    for (int k = 0; k < 3; ++k) { H.qmin[k] = B.qmin[k]; H.qstep[k] = B.qstep[k]; H.bmin[k] = B.bmin[k]; H.bmax[k] = B.bmax[k]; }
    H.build_ms = scene->info.build_ms;
    std::memcpy(p, &H, sizeof(H));
    size_t off = sizeof(H);
    for (const HostObject& o : scene->hs.objects) {
        ExportObject E{};
        put3(E.emitted, o.emitted); put3(E.k, o.k); put3(E.color_d, o.color_d); put3(E.color_s, o.color_s); put3(E.pos, o.pos); put3(E.n, o.n);
        put3(E.bb_min, o.bb_min); put3(E.bb_max, o.bb_max);
        E.phong_kd = o.phong_kd; E.phong_ks = o.phong_ks; E.r = o.r; E.surface_area = o.surface_area;
        E.brdf = o.brdf; E.phong_power = o.phong_power; E.geom = o.geom;
        E.n_vertices = o.vertices.size(); E.n_indices = o.indices.size(); E.n_cum = o.cumulative_area.size();
        std::memcpy(p + off, &E, sizeof(E)); off += sizeof(E);
        for (const D3& v : o.vertices) { const double t[3] = {v.x, v.y, v.z}; std::memcpy(p + off, t, sizeof(t)); off += sizeof(t); }
        if (!o.indices.empty()) { std::memcpy(p + off, o.indices.data(), o.indices.size() * sizeof(uint32_t)); off += o.indices.size() * sizeof(uint32_t); }
        if (!o.cumulative_area.empty()) { std::memcpy(p + off, o.cumulative_area.data(), o.cumulative_area.size() * sizeof(double)); off += o.cumulative_area.size() * sizeof(double); }
    }
    if (off < lbvh_off) std::memset(p + off, 0, lbvh_off - off);   // alignment gap: the blob is a pure function of the scene
    if (n_tris) {
        CU_TRY(cudaSetDevice(scene->device));
        off = lbvh_off;
        auto down = [&](const void* src, size_t bytes) { cudaError_t e = cudaMemcpy(p + off, src, bytes, cudaMemcpyDeviceToHost); off += bytes; return e; };
        CU_TRY(down(B.d_nodes, (size_t)B.n_nodes * 4 * sizeof(float4)));
        CU_TRY(down(B.d_qnodes, (size_t)B.n_nodes * 2 * sizeof(uint4)));
        CU_TRY(down(B.d_tris, (size_t)n_tris * TRI_STRIDE * sizeof(float4)));
        CU_TRY(down(B.d_tri_nrm, (size_t)n_tris * sizeof(float4)));
    }
    return (int64_t)total;
}

int rtb_scene_import(const void* buf, int64_t bytes, int device, rtb_scene** out) {
    if (!buf || !out) return fail(RTB_EINVAL, "NULL argument");
    *out = nullptr;
    const unsigned char* p = static_cast<const unsigned char*>(buf);
    ExportHeader H;
    if (bytes < (int64_t)sizeof(H)) return fail(RTB_EPARSE, "exported scene: truncated header");
    std::memcpy(&H, p, sizeof(H));
    if (std::memcmp(H.magic, EXPORT_MAGIC, 8) != 0 || H.total_bytes != (uint64_t)bytes || H.n_objects < 0 || H.n_objects > MAX_OBJECTS)
        return fail(RTB_EPARSE, "exported scene: bad magic, size or object count");
    rtb_scene* sc = new rtb_scene();
    sc->device = device;
    sc->hs.cam_pos = get3(H.cam_pos);
    sc->hs.cam_dir = get3(H.cam_dir);
    sc->hs.light = H.light;
    size_t off = sizeof(H);
    auto need = [&](size_t n) { return off + n <= (size_t)bytes; };
    for (int i = 0; i < H.n_objects; ++i) {
        ExportObject E;
        if (!need(sizeof(E))) { delete sc; return fail(RTB_EPARSE, "exported scene: truncated object table"); }
        std::memcpy(&E, p + off, sizeof(E)); off += sizeof(E);
        if (E.n_vertices > (1ull << 31) || E.n_indices > (1ull << 32) || E.n_cum > (1ull << 31) ||
            !need(E.n_vertices * 24 + E.n_indices * 4 + E.n_cum * 8)) { delete sc; return fail(RTB_EPARSE, "exported scene: truncated mesh data"); }
        HostObject o;
        o.emitted = get3(E.emitted); o.k = get3(E.k); o.color_d = get3(E.color_d); o.color_s = get3(E.color_s); o.pos = get3(E.pos); o.n = get3(E.n);
        o.bb_min = get3(E.bb_min); o.bb_max = get3(E.bb_max);
        o.phong_kd = E.phong_kd; o.phong_ks = E.phong_ks; o.r = E.r; o.surface_area = E.surface_area;
        o.brdf = E.brdf; o.phong_power = E.phong_power; o.geom = E.geom;
        o.vertices.resize((size_t)E.n_vertices);
        for (D3& v : o.vertices) { double t[3]; std::memcpy(t, p + off, sizeof(t)); off += sizeof(t); v = D3{t[0], t[1], t[2]}; }
        o.indices.resize((size_t)E.n_indices);
        if (E.n_indices) { std::memcpy(o.indices.data(), p + off, (size_t)E.n_indices * 4); off += (size_t)E.n_indices * 4; }
        o.cumulative_area.resize((size_t)E.n_cum);
        if (E.n_cum) { std::memcpy(o.cumulative_area.data(), p + off, (size_t)E.n_cum * 8); off += (size_t)E.n_cum * 8; }
        sc->hs.objects.push_back(std::move(o));
    }
    off = align_up(off, 16);
    LbvhImport imp{};
    imp.n_tris = H.n_tris;
    LbvhResult& M = imp.meta;
    M.n_nodes = H.n_nodes; M.n_leaves = H.n_leaves; M.root = H.root; M.depth = H.depth;
    for (int k = 0; k < 3; ++k) { M.qmin[k] = H.qmin[k]; M.qstep[k] = H.qstep[k]; M.bmin[k] = H.bmin[k]; M.bmax[k] = H.bmax[k]; }
    if (H.n_tris > 0) {
        if (H.n_nodes < 0 || !need(lbvh_bytes(M, H.n_tris))) { delete sc; return fail(RTB_EPARSE, "exported scene: truncated LBVH tables"); }
        imp.nodes = reinterpret_cast<const float4*>(p + off); off += (size_t)M.n_nodes * 4 * sizeof(float4);
        imp.qnodes = reinterpret_cast<const uint4*>(p + off); off += (size_t)M.n_nodes * 2 * sizeof(uint4);
        imp.tris = reinterpret_cast<const float4*>(p + off); off += (size_t)H.n_tris * TRI_STRIDE * sizeof(float4);
        imp.tri_nrm = reinterpret_cast<const float4*>(p + off);
    }
    int rc = finish_scene(sc, RTB_OK, std::string(), out, H.n_tris >= 0 ? &imp : nullptr);   // no tables in the blob: build here
    if (rc == RTB_OK && H.n_tris >= 0) (*out)->info.build_ms = H.build_ms;   // the build happened on the exporting rank
    return rc;
}

void rtb_scene_destroy(rtb_scene* scene) { delete scene; }

int rtb_scene_get_info(const rtb_scene* scene, rtb_scene_info* info) {
    if (!scene || !info) return fail(RTB_EINVAL, "NULL argument");
    *info = scene->info;
    return RTB_OK;
}

int rtb_scene_upload(rtb_scene* scene, uint64_t* bytes) {
    if (int rc = need_device(scene)) return rc;
    return upload_scene(scene, bytes);
}

int64_t rtb_scene_triangles(const rtb_scene* scene, float* out9, int64_t cap) {
    if (!scene) return fail(RTB_EINVAL, "NULL scene");
    int64_t n = (int64_t)scene->fs.tri_obj.size();
    if (out9 && cap > 0) std::memcpy(out9, scene->fs.tri_verts.data(), (size_t)std::min(n, cap) * 9 * sizeof(float));
    return n;
}

int64_t rtb_scene_lights(const rtb_scene* scene, int32_t* objects, double* prob, double* area, int64_t cap) {
    if (!scene) return fail(RTB_EINVAL, "NULL scene");
    const std::vector<FlatLight>& L = scene->fs.lights;
    for (int64_t k = 0; k < std::min<int64_t>((int64_t)L.size(), cap); ++k) {
        if (objects) objects[k] = L[(size_t)k].obj;
        if (prob) prob[k] = L[(size_t)k].prob;
        if (area) area[k] = L[(size_t)k].area;
    }
    return (int64_t)L.size();
}

int rtb_scene_object(const rtb_scene* scene, int32_t index, rtb_object_info* out) {
    if (!scene || !out) return fail(RTB_EINVAL, "NULL argument");
    if (index < 0 || index >= scene->fs.n_objects) return fail(RTB_EINVAL, "object index out of range");
    const HostObject& o = scene->hs.objects[index];
    std::memset(out, 0, sizeof(*out));
    out->brdf = o.brdf;
    out->geometry = o.geom;
    out->emitted[0] = o.emitted.x; out->emitted[1] = o.emitted.y; out->emitted[2] = o.emitted.z;
    if (o.brdf == BRDF_PHONG) {
        out->k[0] = o.phong_kd; out->k[1] = o.phong_ks; out->k[2] = o.phong_power;
        out->color_d[0] = o.color_d.x; out->color_d[1] = o.color_d.y; out->color_d[2] = o.color_d.z;
        out->color_s[0] = o.color_s.x; out->color_s[1] = o.color_s.y; out->color_s[2] = o.color_s.z;
    } else if (o.brdf == BRDF_DIELECTRIC) {
        out->k[0] = o.k.x; out->k[1] = scene->fs.materials[index].k[1];   // ior, orientation sign
        out->color_d[0] = o.color_d.x; out->color_d[1] = o.color_d.y; out->color_d[2] = o.color_d.z;
    } else {
        out->k[0] = o.k.x; out->k[1] = o.k.y; out->k[2] = o.k.z;
    }
    out->pos[0] = o.pos.x; out->pos[1] = o.pos.y; out->pos[2] = o.pos.z;
    out->n[0] = o.n.x; out->n[1] = o.n.y; out->n[2] = o.n.z;
    out->r = o.r;
    out->n_triangles = (int32_t)(o.indices.size() / 3);
    out->first_triangle = scene->fs.materials[index].first_tri;
    out->bb_min[0] = o.bb_min.x; out->bb_min[1] = o.bb_min.y; out->bb_min[2] = o.bb_min.z;
    out->bb_max[0] = o.bb_max.x; out->bb_max[1] = o.bb_max.y; out->bb_max[2] = o.bb_max.z;
    out->surface_area = o.surface_area;
    return RTB_OK;
}

int64_t rtb_local_pixels(const rtb_params* params) {
    if (check_params(params) != RTB_OK) return RTB_EINVAL;
    return (int64_t)local_tiles(params) * 1024;
}

int64_t rtb_tile_map(const rtb_params* params, int32_t* xy, int64_t cap) {
    if (check_params(params) != RTB_OK) return RTB_EINVAL;
    int64_t n = (int64_t)local_tiles(params) * 1024;
    int tiles_x = (params->width + TILE - 1) / TILE;
    for (int64_t lp = 0; lp < n && lp < cap && xy; ++lp) {
        int x, y;
        bool in = local_to_xy((int)lp, params->rank, params->world, tiles_x, params->width, params->height, x, y);
        xy[2 * lp] = in ? x : -1;
        xy[2 * lp + 1] = in ? y : -1;
    }
    return n;
}

int rtb_get_stats(const rtb_scene* scene, rtb_stats* stats) {
    if (!scene || !stats) return fail(RTB_EINVAL, "NULL argument");
    if (g_thread_stats_scene == scene) {   // this thread has rendered on the scene: its own last call, whatever other threads did since
        *stats = g_thread_stats;
        return RTB_OK;
    }
    rtb_scene* s = const_cast<rtb_scene*>(scene);
    std::lock_guard<std::mutex> lk(s->mu);
    *stats = s->last_stats;
    return RTB_OK;
}

int rtb_render_device(rtb_scene* scene, const rtb_params* params, void* d_rgb8_tiles, void* d_subpixel_sums, volatile int* cancel) {
    if (int rc0 = need_device(scene)) return rc0;
    int rc = check_params(params);
    if (rc != RTB_OK) return rc;
    if ((rc = need_accel(scene, params)) != RTB_OK) return rc;
    RenderContext* c = acquire_context(scene, default_pool(params));
    RenderArgs a;
    rtb_stats st{};
    bool cancelled = false;
    rc = render_into_context(scene, params, c, a, cancel, st, cancelled);
    if (rc == RTB_OK && !cancelled && d_rgb8_tiles)
        rc = resolve_to(c, a, (unsigned char*)d_rgb8_tiles, (float4*)d_subpixel_sums, 0, st);
    publish_stats(scene, st);
    release_context(scene, c);
    if (rc != RTB_OK) return rc;
    return cancelled ? RTB_ECANCELLED : RTB_OK;
}

int rtb_render(rtb_scene* scene, const rtb_params* params, uint8_t* rgb8_out, volatile int* cancel) {
    if (!scene || !rgb8_out) return fail(RTB_EINVAL, "NULL argument");
    if (int rc0 = need_device(scene)) return rc0;
    int rc = check_params(params);
    if (rc != RTB_OK) return rc;
    if ((rc = need_accel(scene, params)) != RTB_OK) return rc;
    RenderContext* c = acquire_context(scene, default_pool(params));
    RenderArgs a;
    rtb_stats st{};
    bool cancelled = false;
    rc = render_into_context(scene, params, c, a, cancel, st, cancelled);
    if (rc == RTB_OK && !cancelled) {
        const size_t frame = (size_t)params->width * params->height * 3;
        const bool whole = params->world == 1;
        const size_t bytes = whole ? frame : (size_t)a.n_local_tiles * 1024 * 3;
        rc = ensure_rgb(c, std::max<size_t>(bytes, 1), true);
        if (rc == RTB_OK) rc = resolve_to(c, a, c->d_rgb, nullptr, whole ? 1 : 0, st);
        if (rc == RTB_OK && bytes) {
            cudaError_t e = cudaMemcpyAsync(c->h_rgb, c->d_rgb, bytes, cudaMemcpyDeviceToHost, c->stream);
            if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
            if (e != cudaSuccess) rc = fail(RTB_ECUDA, std::string("frame read-back: ") + cudaGetErrorString(e));
        }
        if (rc == RTB_OK) {
            if (whole) std::memcpy(rgb8_out, c->h_rgb, frame);
            else {
                // tile order walks 8x4-pixel blocks: 8 consecutive slots are 8 consecutive pixels of one row
                for (int lp = 0; lp < a.n_local_tiles * 1024; lp += 8) {
                    int x, y;
                    if (!local_to_xy(lp, a.rank, a.world, a.tiles_x, a.width, a.height, x, y)) continue;
                    const int run = std::min(8, a.width - x);
                    std::memcpy(rgb8_out + ((size_t)y * a.width + x) * 3, c->h_rgb + (size_t)lp * 3, (size_t)run * 3);
                }
            }
        }
    }
    publish_stats(scene, st);
    release_context(scene, c);
    if (rc != RTB_OK) return rc;
    return cancelled ? RTB_ECANCELLED : RTB_OK;
}

int rtb_render_adaptive(rtb_scene* scene, const rtb_params* params, const rtb_adaptive* opts, uint8_t* rgb8_out, int32_t* tile_spp,
                        float* tile_error, volatile int* cancel) {
    if (!scene || !rgb8_out) return fail(RTB_EINVAL, "NULL argument");
    int rc = check_params(params);
    if (rc == RTB_OK) rc = check_adaptive(params, opts);
    if (rc != RTB_OK) return rc;
    return render_whole_frame(scene, params, opts, nullptr, rgb8_out, tile_spp, tile_error, cancel);
}

int rtb_render_denoised(rtb_scene* scene, const rtb_params* params, const rtb_adaptive* adaptive, const rtb_denoise* denoise,
                        uint8_t* rgb8_out, int32_t* tile_spp, float* tile_error, volatile int* cancel) {
    if (!scene || !rgb8_out) return fail(RTB_EINVAL, "NULL argument");
    int rc = check_params(params);
    if (rc == RTB_OK && adaptive) rc = check_adaptive(params, adaptive);
    if (rc == RTB_OK) rc = check_denoise(params, denoise);
    if (rc != RTB_OK) return rc;
    return render_whole_frame(scene, params, adaptive, denoise, rgb8_out, tile_spp, tile_error, cancel);
}

int rtb_scene_gbuffer(rtb_scene* scene, int32_t width, int32_t height, int32_t accel, float* albedo3, float* normal3, float* depth,
                      int32_t* obj) {
    if (!scene) return fail(RTB_EINVAL, "NULL scene");
    if (width <= 0 || height <= 0 || width > 65535 || height > 65535 || (long long)width * height >= (1ll << 31))
        return fail(RTB_EINVAL, "width/height must be in 1..65535");
    if (accel != RTB_ACCEL_LBVH && accel != RTB_ACCEL_OCTREE_REFERENCE) return fail(RTB_EINVAL, "unknown accel mode");
    if (int rc0 = need_device(scene)) return rc0;
    rtb_params p{};
    p.accel = accel;
    if (int rc1 = need_accel(scene, &p)) return rc1;
    const size_t pixels = (size_t)width * height;
    RenderContext* c = acquire_context(scene);
    int rc = ensure_context(scene, c, 1024, 1024, 0);
    if (rc == RTB_OK) rc = ensure_denoise(c, pixels);
    if (rc == RTB_OK) rc = launch_gbuffer(scene, c, width, height, accel, c->stream);
    std::vector<float4> host(pixels * 2);
    if (rc == RTB_OK) {
        cudaError_t e = cudaMemcpyAsync(host.data(), c->dn_guides, pixels * 2 * sizeof(float4), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) rc = fail(RTB_ECUDA, std::string("rtb_scene_gbuffer: ") + cudaGetErrorString(e));
    }
    release_context(scene, c);
    if (rc != RTB_OK) return rc;
    for (size_t i = 0; i < pixels; ++i) {
        const float4 ga = host[i], gn = host[pixels + i];
        if (albedo3) { albedo3[3 * i] = ga.x; albedo3[3 * i + 1] = ga.y; albedo3[3 * i + 2] = ga.z; }
        if (normal3) { normal3[3 * i] = gn.x; normal3[3 * i + 1] = gn.y; normal3[3 * i + 2] = gn.z; }
        if (depth) depth[i] = ga.w;
        if (obj) std::memcpy(&obj[i], &gn.w, 4);
    }
    return RTB_OK;
}

int rtb_denoise_image(int device, int32_t width, int32_t height, const rtb_denoise* denoise, const float* color3, const float* variance,
                      const float* albedo3, const float* normal3, const float* depth, const int32_t* obj, float* out3) {
    int rc = check_denoise(nullptr, denoise);
    if (rc != RTB_OK) return rc;
    if (!color3 || !variance || !albedo3 || !normal3 || !depth || !obj || !out3) return fail(RTB_EINVAL, "NULL argument");
    if (width <= 0 || height <= 0 || (long long)width * height >= (1ll << 31)) return fail(RTB_EINVAL, "bad image size");
    const size_t pixels = (size_t)width * height;
    std::vector<float4> host(pixels * 3);   // guides (albedo | depth, normal | object), then colour | variance
    for (size_t i = 0; i < pixels; ++i) {
        float o;
        std::memcpy(&o, &obj[i], 4);
        host[i] = make_float4(albedo3[3 * i], albedo3[3 * i + 1], albedo3[3 * i + 2], depth[i]);
        host[pixels + i] = make_float4(normal3[3 * i], normal3[3 * i + 1], normal3[3 * i + 2], o);
        host[2 * pixels + i] = make_float4(color3[3 * i], color3[3 * i + 1], color3[3 * i + 2], variance[i]);
    }
    CU_TRY(cudaSetDevice(device));
    float4 *d_guides = nullptr, *d_buf = nullptr;
    float* d_out = nullptr;
    cudaStream_t st = nullptr;
    cudaError_t e = cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking);
    auto T = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    T(cudaMalloc((void**)&d_guides, pixels * 2 * sizeof(float4)));
    T(cudaMalloc((void**)&d_buf, pixels * 2 * sizeof(float4)));
    T(cudaMalloc((void**)&d_out, pixels * 3 * sizeof(float)));
    T(cudaMemcpyAsync(d_guides, host.data(), pixels * 2 * sizeof(float4), cudaMemcpyHostToDevice, st));
    T(cudaMemcpyAsync(d_buf + pixels, host.data() + 2 * pixels, pixels * sizeof(float4), cudaMemcpyHostToDevice, st));
    if (e == cudaSuccess) {
        DenoiseArgs d{};
        d.width = width;
        d.height = height;
        d.ga = d_guides;
        d.gn = d_guides + pixels;
        d.buf[0] = d_buf;
        d.buf[1] = d_buf + pixels;   // d.accum = nullptr: k_denoise_prep reads the colour and variance from here
        launch_filter(d, *denoise, nullptr, d_out, st);
        T(cudaGetLastError());
    }
    T(cudaMemcpyAsync(out3, d_out, pixels * 3 * sizeof(float), cudaMemcpyDeviceToHost, st));
    T(cudaStreamSynchronize(st));
    cudaFree(d_guides); cudaFree(d_buf); cudaFree(d_out);
    if (st) cudaStreamDestroy(st);
    if (e != cudaSuccess) return fail(RTB_ECUDA, std::string("rtb_denoise_image: ") + cudaGetErrorString(e));
    return RTB_OK;
}

int rtb_untile_device_async(const rtb_params* params, const void* d_shards, int64_t shard_stride, void* d_rgb8_frame, int device,
                            void* cuda_stream) {
    int rc = check_params(params);
    if (rc != RTB_OK) return rc;
    if (!d_shards || !d_rgb8_frame) return fail(RTB_EINVAL, "NULL argument");
    CU_TRY(cudaSetDevice(device));
    int tx = (params->width + TILE - 1) / TILE, ty = (params->height + TILE - 1) / TILE;
    long long total = (long long)tx * ty * 1024;
    k_untile<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)cuda_stream>>>((const unsigned char*)d_shards, shard_stride, params->world,
                                                                                    tx, ty, params->width, params->height,
                                                                                    (unsigned char*)d_rgb8_frame);
    CU_TRY(cudaGetLastError());
    return RTB_OK;
}

int rtb_untile_device(const rtb_params* params, const void* d_shards, int64_t shard_stride, void* d_rgb8_frame, int device) {
    int rc = rtb_untile_device_async(params, d_shards, shard_stride, d_rgb8_frame, device, nullptr);
    if (rc != RTB_OK) return rc;
    CU_TRY(cudaStreamSynchronize(nullptr));   // legacy default stream only — not the whole device
    return RTB_OK;
}

// ---------------------------------------------------------------- parity hooks
static int trace_common(rtb_scene* scene, int64_t n, const float* org3, const float* dir3, int width, int height, int sx, int sy,
                        float dx, float dy, int32_t* obj, int32_t* tri, float* t, uint64_t* work2, int accel = RTB_ACCEL_LBVH) {
    if (!scene || !obj || !tri || !t) return fail(RTB_EINVAL, "NULL argument");
    if (int rc0 = need_device(scene)) return rc0;
    if (accel != RTB_ACCEL_LBVH && accel != RTB_ACCEL_OCTREE_REFERENCE) return fail(RTB_EINVAL, "unknown accel mode");
    if (accel == RTB_ACCEL_OCTREE_REFERENCE && scene->view.n_tris > 0)
        if (int rc1 = ensure_octrees(scene)) return rc1;
    if (n <= 0) return RTB_OK;
    CU_TRY(cudaSetDevice(scene->device));
    float *d_org = nullptr, *d_dir = nullptr, *d_t = nullptr;
    int32_t *d_obj = nullptr, *d_tri = nullptr;
    unsigned long long* d_work = nullptr;
    auto cleanup = [&]() { cudaFree(d_org); cudaFree(d_dir); cudaFree(d_t); cudaFree(d_obj); cudaFree(d_tri); cudaFree(d_work); };
    cudaError_t e = cudaSuccess;
    auto T = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
    if (org3) {
        T(cudaMalloc((void**)&d_org, (size_t)n * 3 * sizeof(float)));
        T(cudaMalloc((void**)&d_dir, (size_t)n * 3 * sizeof(float)));
        if (e == cudaSuccess) T(cudaMemcpy(d_org, org3, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice));
        if (e == cudaSuccess) T(cudaMemcpy(d_dir, dir3, (size_t)n * 3 * sizeof(float), cudaMemcpyHostToDevice));
    }
    T(cudaMalloc((void**)&d_t, (size_t)n * sizeof(float)));
    T(cudaMalloc((void**)&d_obj, (size_t)n * sizeof(int32_t)));
    T(cudaMalloc((void**)&d_tri, (size_t)n * sizeof(int32_t)));
    T(cudaMalloc((void**)&d_work, 2 * sizeof(unsigned long long)));
    if (e == cudaSuccess) T(cudaMemset(d_work, 0, 2 * sizeof(unsigned long long)));
    if (e == cudaSuccess) {
        const size_t smem = shared_scene_bytes(scene->view.n_prims, scene->view.n_objects, WF_THREADS);
        Camera cam = make_camera(scene->fs.cam_pos, scene->fs.cam_dir, std::max(width, 1), std::max(height, 1));
        int grid = (int)std::min<int64_t>((n + WF_THREADS - 1) / WF_THREADS, 148 * 8);
        if (work2) {
            T(cudaFuncSetAttribute(k_trace_rays<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shared_scene_bytes(MAX_OBJECTS, MAX_OBJECTS, WF_THREADS)));
            k_trace_rays<true><<<grid, WF_THREADS, smem>>>(scene->view, n, d_org, d_dir, cam, width, height, sx, sy, dx, dy, d_obj, d_tri, d_t, d_work, accel);
        } else {
            T(cudaFuncSetAttribute(k_trace_rays<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shared_scene_bytes(MAX_OBJECTS, MAX_OBJECTS, WF_THREADS)));
            k_trace_rays<false><<<grid, WF_THREADS, smem>>>(scene->view, n, d_org, d_dir, cam, width, height, sx, sy, dx, dy, d_obj, d_tri, d_t, d_work, accel);
        }
        T(cudaDeviceSynchronize());
        T(cudaGetLastError());
    }
    if (e == cudaSuccess) T(cudaMemcpy(obj, d_obj, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (e == cudaSuccess) T(cudaMemcpy(tri, d_tri, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost));
    if (e == cudaSuccess) T(cudaMemcpy(t, d_t, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
    if (e == cudaSuccess && work2) T(cudaMemcpy(work2, d_work, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    cleanup();
    if (e != cudaSuccess) return fail(RTB_ECUDA, std::string("rtb_trace: ") + cudaGetErrorString(e));
    return RTB_OK;
}

int rtb_trace_primary(rtb_scene* scene, int32_t width, int32_t height, int32_t sx, int32_t sy, float dx, float dy, int32_t* obj,
                      int32_t* tri, float* t) {
    if (width <= 0 || height <= 0) return fail(RTB_EINVAL, "bad frame size");
    return trace_common(scene, (int64_t)width * height, nullptr, nullptr, width, height, sx, sy, dx, dy, obj, tri, t, nullptr);
}

int rtb_trace_rays(rtb_scene* scene, int64_t n, const float* org3, const float* dir3, int32_t* obj, int32_t* tri, float* t,
                   uint64_t* work2) {
    if (!org3 || !dir3) return fail(RTB_EINVAL, "NULL rays");
    return trace_common(scene, n, org3, dir3, 1, 1, 0, 0, 0.f, 0.f, obj, tri, t, work2);
}

// host-only: Octree::build for one mesh object — counts[4] = {nodes, parents, leaves, triangle references}; works on
// device = -1 handles too (the loader checks run without a GPU)
int rtb_scene_octree_stats(const rtb_scene* scene, int32_t object, int64_t* counts4) {
    if (!scene || !counts4) return fail(RTB_EINVAL, "NULL argument");
    if (object < 0 || object >= scene->fs.n_objects) return fail(RTB_EINVAL, "object index out of range");
    const HostObject& ob = scene->hs.objects[(size_t)object];
    if (ob.geom != GEOM_MESH) return fail(RTB_EINVAL, "object is not a mesh");
    HostOctree ot;
    build_reference_octree(ob, ot);
    int64_t parents = 0, leaves = 0;
    for (const HostOctreeNode& n : ot.nodes) (n.count < 0 ? parents : leaves)++;
    counts4[0] = (int64_t)ot.nodes.size();
    counts4[1] = parents;
    counts4[2] = leaves;
    counts4[3] = (int64_t)ot.tri_refs.size();
    return RTB_OK;
}

int rtb_trace_rays_accel(rtb_scene* scene, int32_t accel, int64_t n, const float* org3, const float* dir3, int32_t* obj, int32_t* tri, float* t) {
    if (!org3 || !dir3) return fail(RTB_EINVAL, "NULL rays");
    return trace_common(scene, n, org3, dir3, 1, 1, 0, 0, 0.f, 0.f, obj, tri, t, nullptr, accel);
}

int rtb_sample_radiance(rtb_scene* scene, const rtb_params* params, int64_t n, const int32_t* px, const int32_t* py,
                        const int32_t* sample_idx, float* rgb3) {
    if (!scene || !px || !py || !sample_idx || !rgb3) return fail(RTB_EINVAL, "NULL argument");
    if (int rc0 = need_device(scene)) return rc0;
    int rc = check_params(params);
    if (rc != RTB_OK) return rc;
    if ((rc = need_accel(scene, params)) != RTB_OK) return rc;
    if (n <= 0) return RTB_OK;
    if (params->spp < 4) return fail(RTB_EINVAL, "spp < 4 has no samples");
    for (int64_t i = 0; i < n; ++i)
        if (px[i] < 0 || px[i] >= params->width || py[i] < 0 || py[i] >= params->height || sample_idx[i] < 0 ||
            sample_idx[i] >= params->spp / 4 * 4)
            return fail(RTB_EINVAL, "probe item out of range");
    RenderContext* c = acquire_context(scene);
    uint32_t P = (uint32_t)std::min<int64_t>(std::max<int64_t>((n + 31) / 32 * 32, 1024), 1 << 22);
    uint32_t SP = shadow_slots(params->estimator, P);
    rc = ensure_context(scene, c, P, SP, (size_t)n);
    RenderArgs a;
    rtb_stats st{};
    if (rc == RTB_OK) {
        if (c->probe_cap < (size_t)n * 3) {
            cudaFree(c->d_probe);
            c->d_probe = nullptr;
            if (cudaMalloc((void**)&c->d_probe, (size_t)n * 3 * sizeof(int32_t)) != cudaSuccess) rc = fail(RTB_ECUDA, "probe alloc");
            else c->probe_cap = (size_t)n * 3;
        }
    }
    if (rc == RTB_OK) {
        fill_args(scene, params, c, a);
        a.probe_px = c->d_probe;
        a.probe_py = c->d_probe + n;
        a.probe_sample = c->d_probe + 2 * n;
        a.n_probe = (int)n;
        cudaError_t e = cudaMemcpyAsync(c->d_probe, px, n * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_probe + n, py, n * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_probe + 2 * n, sample_idx, n * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->accum, 0, (size_t)n * sizeof(float4), c->stream);
        if (e != cudaSuccess) rc = fail(RTB_ECUDA, cudaGetErrorString(e));
    }
    bool cancelled = false;
    if (rc == RTB_OK) rc = run_wavefront(scene, c, a, 0, 0, params->tuning[0] == 1, nullptr, st, cancelled);
    if (rc == RTB_OK) {
        std::vector<float4> host((size_t)n);
        cudaError_t e = cudaMemcpy(host.data(), c->accum, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost);
        if (e != cudaSuccess) rc = fail(RTB_ECUDA, cudaGetErrorString(e));
        else
            for (int64_t i = 0; i < n; ++i) {
                rgb3[3 * i] = host[i].x; rgb3[3 * i + 1] = host[i].y; rgb3[3 * i + 2] = host[i].z;
            }
    }
    publish_stats(scene, st);
    release_context(scene, c);
    return rc;
}

// sample_pixel (src/server.rs:320-364) for a LIST of pixels: the full sample set of every listed pixel, resolved to the Vec3
// the reference's function returns (gamma-corrected, 0..255.5, before RenderJob::run's `as u8`).  Same RNG counters as a frame.
int rtb_sample_pixels(rtb_scene* scene, const rtb_params* params, int64_t n, const int32_t* px, const int32_t* py, float* rgb3) {
    if (!scene || !px || !py || !rgb3) return fail(RTB_EINVAL, "NULL argument");
    if (int rc0 = need_device(scene)) return rc0;
    int rc = check_params(params);
    if (rc != RTB_OK) return rc;
    if ((rc = need_accel(scene, params)) != RTB_OK) return rc;
    if (n <= 0) return RTB_OK;
    if (n > (1 << 24)) return fail(RTB_EINVAL, "at most 2^24 pixels per call");
    for (int64_t i = 0; i < n; ++i)
        if (px[i] < 0 || px[i] >= params->width || py[i] < 0 || py[i] >= params->height) return fail(RTB_EINVAL, "pixel out of range");
    const int num_samples = params->spp / 4;
    RenderContext* c = acquire_context(scene);
    const uint64_t samples = (uint64_t)n * 4ull * (uint64_t)std::max(1, num_samples);
    const uint32_t P = pool_for(samples, params->pool_paths);
    const uint32_t SP = shadow_slots(params->estimator, P);
    rc = ensure_context(scene, c, P, SP, (size_t)n * 4, requested_bin_bits(scene, params) > 0);
    RenderArgs a;
    rtb_stats st{};
    float* d_out = nullptr;
    if (rc == RTB_OK && c->probe_cap < (size_t)n * 3) {
        cudaFree(c->d_probe);
        c->d_probe = nullptr;
        c->probe_cap = 0;
        if (cudaMalloc((void**)&c->d_probe, (size_t)n * 3 * sizeof(int32_t)) != cudaSuccess) rc = fail(RTB_ECUDA, "probe alloc");
        else c->probe_cap = (size_t)n * 3;
    }
    if (rc == RTB_OK) {
        fill_args(scene, params, c, a);
        a.probe_px = c->d_probe;
        a.probe_py = c->d_probe + n;
        a.probe_sample = nullptr;
        a.n_probe = (int)n;
        a.pixel_list = 1;
        cudaError_t e = cudaMemcpyAsync(c->d_probe, px, n * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = cudaMemcpyAsync(c->d_probe + n, py, n * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream);
        if (e == cudaSuccess) e = cudaMemsetAsync(c->accum, 0, (size_t)n * 4 * sizeof(float4), c->stream);
        if (e != cudaSuccess) rc = fail(RTB_ECUDA, cudaGetErrorString(e));
    }
    bool cancelled = false;
    if (rc == RTB_OK && num_samples > 0) rc = run_wavefront(scene, c, a, 0u, (uint32_t)num_samples * 4u, false, nullptr, st, cancelled);
    if (rc == RTB_OK) {
        // the pixel list is no longer needed: the result overwrites it (n x 3 floats in the 3n-word probe buffer)
        d_out = reinterpret_cast<float*>(c->d_probe);
        k_resolve_list<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->accum, (int)n, num_samples, d_out);
        cudaError_t e = cudaMemcpyAsync(rgb3, d_out, (size_t)n * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        if (e != cudaSuccess) rc = fail(RTB_ECUDA, cudaGetErrorString(e));
        st.kernel_launches += 1;
    }
    publish_stats(scene, st);
    release_context(scene, c);
    return rc;
}

int rtb_fp32_peak(int device, double* tflops) {
    if (!tflops) return fail(RTB_EINVAL, "NULL argument");
    CU_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU_TRY(cudaGetDeviceProperties(&prop, device));
    const int threads = 256, blocks = prop.multiProcessorCount * 8, iters = 4096;
    float* d = nullptr;
    CU_TRY(cudaMalloc((void**)&d, (size_t)threads * blocks * sizeof(float)));
    cudaEvent_t e0, e1;
    CU_TRY(cudaEventCreate(&e0));
    CU_TRY(cudaEventCreate(&e1));
    double best = 0;
    for (int rep = 0; rep < 5; ++rep) {
        CU_TRY(cudaEventRecord(e0));
        k_fma_peak<<<blocks, threads>>>(d, iters);
        CU_TRY(cudaEventRecord(e1));
        CU_TRY(cudaEventSynchronize(e1));
        float ms = 0;
        CU_TRY(cudaEventElapsedTime(&ms, e0, e1));
        double flops = 2.0 * 64.0 * iters * (double)threads * blocks;
        best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    *tflops = best;
    return RTB_OK;
}

}  // extern "C"

// ======================================================================================= jobs
// RenderJob::run's message loop (src/server.rs:166-194).  The reference sends every 60-pixel window the moment it is
// sampled; a GPU renders a whole frame region at once, so a streaming job renders the frame in BANDS of whole tile rows,
// top-down, and hands each band to the consumer while the next ones are still being rendered:
//   * worker threads (two when there are enough bands, each with its own render context and stream, so that the
//     under-filled tail iterations of one band overlap the full ones of the next) take bands from a counter, render
//     them into their accumulators and launch resolve + cudaMemcpyAsync into the job's PINNED frame on the context's
//     side stream; a host callback on that stream publishes the band.  The render stream never waits for the copy.
//   * the consumer walks rows top-down in 60-pixel windows straight out of the pinned frame; it takes the job's
//     mutex once per band (when it runs out of published rows), not per record, and nothing is copied twice.
//   * progressive jobs (passes > 1, not in the reference) keep the whole frame as one band per pass and ping-pong
//     between two pinned frames: pass n + 1 renders while pass n is copied and consumed.
struct rtb_job {
    rtb_scene* scene = nullptr;
    rtb_params params{};
    int passes = 1;
    rtb_adaptive adaptive{};   // pass_spp > 0: adaptive job (passes = the most the budget allows; the device decides how many run)
    bool converged = false;    // adaptive job: no tile was left active, the frame is final (guarded by mu)
    bool denoise = false;      // every published frame goes through the denoiser (`dn`) instead of k_resolve; one band
    rtb_denoise dn{};
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv;
    uint8_t* h_frame[2] = {nullptr, nullptr};   // pinned; single pass: [0] only
    size_t frame_bytes = 0;
    cudaEvent_t ev_resolved[2] = {nullptr, nullptr};
    // A band / pass is PUBLISHED (under mu) as soon as its resolve + copy have been enqueued on the side stream, together
    // with an event recorded behind the copy; the consumer waits for that event before it reads the pinned rows.  (Host
    // callbacks on the stream were measured first: their dispatch latency alone capped progressive mode at ~600 frames/s.)
    std::vector<cudaEvent_t> band_copied;   // single pass: one per band
    cudaEvent_t pass_copied[2] = {nullptr, nullptr};
    // single pass: band b covers tile rows [band_ty[b], band_ty[b + 1])
    int n_bands = 1;
    std::vector<int> band_ty;
    std::vector<char> band_done;        // guarded by mu: published
    int bands_synced = 0;               // consumer only: bands whose copy it has waited for
    std::atomic<int> next_band{0};
    // progressive: pass index held by h_frame[b], -1 = free (guarded by mu)
    int buf_pass[2] = {-1, -1};
    int passes_done = 0;
    // consumer side (one thread)
    int pass_consumed = 0, cursor_x = 0, cursor_y = 0, avail_rows = 0;
    const uint8_t* cur = nullptr;
    std::atomic<double> stats_first_ms{-1.0};   // host time until the consumer held its first rows
    volatile int cancel = 0;
    int error = RTB_OK;
    std::string error_msg;
    int workers_running = 0;
    bool finished = false;
    rtb_stats stats{};                  // summed over finished bands / passes (guarded by mu)
    std::chrono::steady_clock::time_point t_begin;
};

namespace {

constexpr int PIXELS_PER_MSG = 60;  // RenderJob::PIXELS_PER_MSG, src/server.rs:145
// Band schedule of a single-pass job: the first bands are small, so the first records leave early; later bands grow,
// because every band pays for its own tail of under-filled wavefront iterations (sizes in samples for a large frame: 8 Mi,
// 8 Mi, 16 Mi, 32 Mi, then 64 Mi each; smaller frames start at a sixteenth of their samples, rtb_job_begin)
constexpr uint64_t BAND_MIN_SAMPLES = 8ull << 20;
constexpr int BAND_GROWTH_CAP = 8;   // largest band = BAND_GROWTH_CAP x the first

double ms_since(const std::chrono::steady_clock::time_point& t0) {
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
}

void add_stats(rtb_stats& d, const rtb_stats& s) {
    d.samples += s.samples; d.rays_primary += s.rays_primary; d.rays_extension += s.rays_extension; d.rays_shadow += s.rays_shadow;
    d.iterations += s.iterations; d.kernel_launches += s.kernel_launches; d.bvh_node_visits += s.bvh_node_visits;
    d.bvh_tri_tests += s.bvh_tri_tests; d.render_ms += s.render_ms; d.extend_ms += s.extend_ms; d.bin_ms += s.bin_ms;
    d.generate_ms += s.generate_ms; d.resolve_ms += s.resolve_ms; d.shade_ms += s.shade_ms; d.rays_bvh += s.rays_bvh;
    d.shadow_bvh += s.shadow_bvh; d.paths_queued += s.paths_queued;
}

void publish_band(rtb_job* j, int band) {
    {
        std::lock_guard<std::mutex> lk(j->mu);
        j->band_done[band] = 1;
    }
    j->cv.notify_all();
}

void publish_pass(rtb_job* j, int pass, int buffer) {
    {
        std::lock_guard<std::mutex> lk(j->mu);
        j->buf_pass[buffer] = pass;
        j->passes_done = pass + 1;
    }
    j->cv.notify_all();
}

void job_worker(rtb_job* j, int worker) {
    rtb_scene* sc = j->scene;
    const rtb_params& p = j->params;
    const int tiles_x = (p.width + TILE - 1) / TILE, tiles_y = (p.height + TILE - 1) / TILE;
    const size_t frame = j->frame_bytes;
    const bool progressive = j->passes > 1;
    int band_tile_rows = progressive ? tiles_y : 1;   // the largest band
    for (int b = 0; !progressive && b < j->n_bands; ++b) band_tile_rows = std::max(band_tile_rows, j->band_ty[b + 1] - j->band_ty[b]);
    // samples in flight at once: one band of a single-pass job, one pass of a progressive one
    uint64_t band_samples = (uint64_t)band_tile_rows * tiles_x * 1024ull * 4ull * (uint64_t)std::max(1, p.spp / 4);
    if (progressive) band_samples = (band_samples + j->passes - 1) / j->passes;
    const uint32_t P = pool_for(band_samples, p.pool_paths);
    const uint32_t SP = shadow_slots(p.estimator, P);
    RenderContext* c = acquire_context(sc, P);
    auto finish = [&](int rc) {
        if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);   // the pinned frame is no longer written by this worker
        release_context(sc, c);
        bool last;
        {
            std::lock_guard<std::mutex> lk(j->mu);
            if (rc != RTB_OK && rc != RTB_ECANCELLED && j->error == RTB_OK) { j->error = rc; j->error_msg = g_last_error; j->cancel = 1; }
            last = --j->workers_running == 0;
            if (last) {
                j->finished = true;
                j->stats.wall_ms = ms_since(j->t_begin);
            }
        }
        if (last) publish_stats(sc, j->stats, false);
        j->cv.notify_all();
    };
    const size_t accum_elems = (size_t)p.width * p.height * 4;
    int rc = ensure_context(sc, c, P, SP, accum_elems, requested_bin_bits(sc, &p) > 0);
    if (rc == RTB_OK) rc = ensure_rgb(c, frame * (progressive ? 2 : 1), false);
    if (rc == RTB_OK && j->denoise) rc = ensure_denoise(c, (size_t)p.width * p.height);
    if (rc == RTB_OK && j->denoise) {   // once: the guides need no RNG.  Complete before any resolve, which may run on copy_stream
        rc = launch_gbuffer(sc, c, p.width, p.height, p.accel, c->stream);
        if (rc == RTB_OK && cudaStreamSynchronize(c->stream) != cudaSuccess) rc = fail(RTB_ECUDA, "streaming job: guides");
    }
    if (rc != RTB_OK) return finish(rc);
    RenderArgs a;
    fill_args(sc, &p, c, a);
    const uint32_t ks_total = (uint32_t)a.num_samples * 4u;
    auto cuda_fail = [&](cudaError_t e) { return finish(fail(RTB_ECUDA, std::string("streaming job: ") + cudaGetErrorString(e))); };

    if (!progressive) {
        for (;;) {
            const int b = j->next_band.fetch_add(1);
            if (b >= j->n_bands) break;
            if (j->cancel) return finish(RTB_ECANCELLED);
            const int ty0 = j->band_ty[b], ty1 = j->band_ty[b + 1];
            const int row0 = ty0 * TILE, row1 = std::min(p.height, ty1 * TILE);
            a.tile_base = ty0 * tiles_x;
            a.n_local_tiles = (ty1 - ty0) * tiles_x;
            cudaError_t e = cudaMemsetAsync(c->accum + (size_t)row0 * p.width * 4, 0, (size_t)(row1 - row0) * p.width * 4 * sizeof(float4), c->stream);
            if (e != cudaSuccess) return cuda_fail(e);
            rtb_stats bs{};
            bool cancelled = false;
            if (ks_total > 0) {
                rc = run_wavefront(sc, c, a, 0u, ks_total, false, &j->cancel, bs, cancelled);   // returns with the band's paths finished
                if (rc != RTB_OK) return finish(rc);
            }
            if (cancelled || j->cancel) return finish(RTB_ECANCELLED);
            // resolve + copy + publish on the side stream; this thread goes straight on to its next band
            const int n = a.n_local_tiles * 1024;
            if (j->denoise) bs.kernel_launches += launch_denoise(c, a, j->dn, c->d_rgb, c->copy_stream) - 1;
            else k_resolve<<<(n + 255) / 256, 256, 0, c->copy_stream>>>(a, c->d_rgb, nullptr, 1);
            const size_t off = (size_t)row0 * p.width * 3, bytes = (size_t)(row1 - row0) * p.width * 3;
            e = cudaMemcpyAsync(j->h_frame[0] + off, c->d_rgb + off, bytes, cudaMemcpyDeviceToHost, c->copy_stream);
            if (e == cudaSuccess) e = cudaEventRecord(j->band_copied[b], c->copy_stream);
            if (e != cudaSuccess) return cuda_fail(e);
            bs.kernel_launches += 1;
            {
                std::lock_guard<std::mutex> lk(j->mu);
                add_stats(j->stats, bs);
            }
            publish_band(j, b);
        }
        return finish(RTB_OK);
    }

    // progressive: one band = the frame; pass n + 1 renders while pass n is copied and consumed
    a.tile_base = 0;
    a.n_local_tiles = tiles_x * tiles_y;
    // resolves pass `pass` (sample counts as `r` gives them) into the pinned frame of its parity and publishes it
    auto publish = [&](int pass, const rtb_stats& ps, const RenderArgs& r) -> int {
        const int b = pass & 1;
        {   // the pinned frame of this parity must have been consumed (passes stay in order, memory stays bounded)
            std::unique_lock<std::mutex> lk(j->mu);
            j->cv.wait(lk, [&] { return j->buf_pass[b] < 0 || j->cancel; });
            if (j->cancel) return RTB_ECANCELLED;
            add_stats(j->stats, ps);
        }
        const int n = a.n_local_tiles * 1024;
        // in stream order: before the next pass adds samples
        if (j->denoise) launch_denoise(c, r, j->dn, c->d_rgb + (size_t)b * frame, c->stream);
        else k_resolve<<<(n + 255) / 256, 256, 0, c->stream>>>(r, c->d_rgb + (size_t)b * frame, nullptr, 1);
        cudaError_t e = cudaEventRecord(j->ev_resolved[b], c->stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(c->copy_stream, j->ev_resolved[b], 0);
        if (e == cudaSuccess) e = cudaMemcpyAsync(j->h_frame[b], c->d_rgb + (size_t)b * frame, frame, cudaMemcpyDeviceToHost, c->copy_stream);
        if (e == cudaSuccess) e = cudaEventRecord(j->pass_copied[b], c->copy_stream);
        if (e != cudaSuccess) return fail(RTB_ECUDA, std::string("streaming job: ") + cudaGetErrorString(e));
        publish_pass(j, pass, b);
        return RTB_OK;
    };
    if (j->adaptive.pass_spp > 0) {
        rtb_stats total{};
        bool cancelled = false;
        rc = run_adaptive(sc, c, a, j->adaptive, &j->cancel, total, cancelled, [&](int pass, const rtb_stats& ps) {
            RenderArgs r = a;
            r.tile_ks = c->ad_tile_ks;   // every tile resolved with its own sample count
            return publish(pass, ps, r);
        });
        if (rc != RTB_OK) return finish(rc);
        if (cancelled || j->cancel) return finish(RTB_ECANCELLED);
        {
            std::lock_guard<std::mutex> lk(j->mu);
            j->converged = true;
        }
        return finish(RTB_OK);
    }
    if (cudaError_t e = cudaMemsetAsync(c->accum, 0, accum_elems * sizeof(float4), c->stream); e != cudaSuccess) return cuda_fail(e);
    const int passes = j->passes;
    for (int pass = 0; pass < passes; ++pass) {
        const uint32_t k0 = (uint32_t)((uint64_t)ks_total * pass / passes), k1 = (uint32_t)((uint64_t)ks_total * (pass + 1) / passes);
        rtb_stats ps{};
        bool cancelled = false;
        if (k1 > k0) {
            rc = run_wavefront(sc, c, a, k0, k1, false, &j->cancel, ps, cancelled);
            if (rc != RTB_OK) return finish(rc);
        }
        if (cancelled || j->cancel) return finish(RTB_ECANCELLED);
        RenderArgs r = a;
        r.ks_done = k1;   // resolve with the per-sub-pixel sample counts reached so far
        if ((rc = publish(pass, ps, r)) != RTB_OK) return finish(rc);
    }
    finish(RTB_OK);
}

// Makes rows [cursor_y, avail_rows) of job->cur readable.  block = false: only looks.  Returns 1 = rows available,
// 0 = the job is complete, RTB_ESTOPPED / negative error, 2 = nothing yet (non-blocking only).
int job_acquire_rows(rtb_job* job, bool block) {
    if (job->cursor_y < job->avail_rows) return 1;
    const bool progressive = job->passes > 1;
    cudaEvent_t copied = nullptr;
    int rows_after = 0;
    {
        std::unique_lock<std::mutex> lk(job->mu);
        const int b = job->pass_consumed & 1;
        const int band = job->bands_synced;   // single pass: the band the cursor is about to enter
        auto ready = [&] {
            return progressive ? job->buf_pass[b] == job->pass_consumed
                               : (job->pass_consumed == 0 && band < job->n_bands && job->band_done[band]);
        };
        // a worker that failed raises `cancel` to stop its peers: the error is reported once they have all stopped
        if (block) job->cv.wait(lk, [&] { return ready() || job->finished || (job->cancel && job->error == RTB_OK); });
        if (job->cancel && job->error == RTB_OK) return RTB_ESTOPPED;
        if (!ready()) {
            if (!job->finished) return 2;
            if (job->error != RTB_OK) return fail(job->error, job->error_msg);
            return 0;
        }
        if (progressive) {
            copied = job->pass_copied[b];
            job->cur = job->h_frame[b];
            rows_after = job->params.height;
        } else {
            copied = job->band_copied[band];
            job->cur = job->h_frame[0];
            rows_after = std::min(job->params.height, job->band_ty[band + 1] * TILE);
        }
    }
    // the copy was enqueued before the band / pass was published: wait for it outside the lock
    if (!block && cudaEventQuery(copied) == cudaErrorNotReady) return 2;
    cudaError_t e = cudaEventSynchronize(copied);
    if (e != cudaSuccess) return fail(RTB_ECUDA, std::string("streaming job: ") + cudaGetErrorString(e));
    if (!progressive) job->bands_synced++;
    job->avail_rows = rows_after;
    if (job->stats_first_ms < 0) job->stats_first_ms = ms_since(job->t_begin);
    return 1;
}

// the consumer has sent the last row of a pass
void job_pass_consumed(rtb_job* job) {
    std::lock_guard<std::mutex> lk(job->mu);
    if (job->passes > 1) job->buf_pass[job->pass_consumed & 1] = -1;
    job->pass_consumed++;
    job->cursor_x = job->cursor_y = 0;
    job->avail_rows = 0;
    job->cv.notify_all();
}


int job_next_record(rtb_job* job, bool block, uint16_t* x, uint16_t* y, uint8_t* n, uint8_t* rgb) {
    const int rc = job_acquire_rows(job, block);
    if (rc != 1) return rc;
    const int w = job->params.width, h = job->params.height;
    int cx = job->cursor_x, cy = job->cursor_y;
    const int cnt = std::min(PIXELS_PER_MSG, w - cx);  // windows(), src/server.rs:254-280
    *x = (uint16_t)cx;
    *y = (uint16_t)cy;
    *n = (uint8_t)cnt;
    std::memcpy(rgb, job->cur + ((size_t)cy * w + cx) * 3, (size_t)cnt * 3);
    cx += cnt;
    if (cx >= w) { cx = 0; ++cy; }
    job->cursor_x = cx;
    job->cursor_y = cy;
    if (cy >= h) job_pass_consumed(job);
    return 1;
}

// adaptive: nullptr for a uniform job; otherwise checked options (check_adaptive) and passes = spp / pass_spp.
// dn: nullptr, or checked options (check_denoise) for a denoised job
int job_begin(rtb_scene* scene, const rtb_params* params, int32_t passes, const rtb_adaptive* adaptive, const rtb_denoise* dn,
              rtb_job** out) {
    if (!scene || !out) return fail(RTB_EINVAL, "NULL argument");
    if (int rc0 = need_device(scene)) return rc0;
    int rc = check_params(params);
    if (rc != RTB_OK) return rc;
    if ((rc = need_accel(scene, params)) != RTB_OK) return rc;
    if (params->world != 1) return fail(RTB_EINVAL, "streaming jobs render whole frames (world must be 1)");
    CU_TRY(cudaSetDevice(scene->device));
    rtb_job* j = new rtb_job();
    j->scene = scene;
    j->params = *params;
    j->passes = std::max(1, passes);
    if (adaptive) j->adaptive = *adaptive;
    if (dn) {
        j->denoise = true;
        j->dn = *dn;
    }
    j->frame_bytes = (size_t)params->width * params->height * 3;
    j->stats.first_record_ms = -1.0;
    const bool progressive = j->passes > 1;
    // bands of whole tile rows (see BAND_MIN_SAMPLES)
    const int tiles_x = (params->width + TILE - 1) / TILE, tiles_y = (params->height + TILE - 1) / TILE;
    const uint64_t row_samples = (uint64_t)tiles_x * 1024ull * 4ull * (uint64_t)std::max(1, params->spp / 4);
    // first band: a sixteenth of the frame's samples, between 1 Mi and BAND_MIN_SAMPLES (8 Mi) — small frames used to wait for a
    // quarter to a half of the whole job before the first record (600x450x256: 22.5 -> 12.5 ms, 600x450x64: 13.3 -> 5.4 ms; job +3 %)
    const uint64_t total_samples = row_samples * (uint64_t)tiles_y;
    uint64_t band_min = std::min<uint64_t>(BAND_MIN_SAMPLES, std::max<uint64_t>(1ull << 20, total_samples / 16));
    if (const char* e = getenv("RTB_BAND_MIN_SAMPLES")) band_min = (uint64_t)std::max(1ll, atoll(e));   // experiment knob
    int rows = (int)std::max<uint64_t>(1, (band_min + row_samples - 1) / row_samples);
    int growth_cap = BAND_GROWTH_CAP;
    if (const char* e = getenv("RTB_BAND_TILE_ROWS")) { rows = std::max(1, atoi(e)); growth_cap = 1; }   // test / experiment knobs
    if (const char* e = getenv("RTB_BAND_GROWTH_CAP")) growth_cap = std::max(1, atoi(e));
    j->band_ty.assign(1, 0);
    if (progressive || j->denoise || 2 * rows > tiles_y) j->band_ty.push_back(tiles_y);   // one band (the denoiser filters whole frames)
    else
        for (int ty = 0, k = 0, mult = 1; ty < tiles_y; ++k) {
            if (k >= 2) mult = std::min(mult * 2, growth_cap);
            ty = std::min(tiles_y, ty + rows * mult);
            if (tiles_y - ty < rows) ty = tiles_y;   // no sliver at the end
            j->band_ty.push_back(ty);
        }
    j->n_bands = (int)j->band_ty.size() - 1;
    j->band_done.assign((size_t)j->n_bands, 0);
    cudaError_t e = cudaMallocHost((void**)&j->h_frame[0], std::max<size_t>(j->frame_bytes, 1));
    if (e == cudaSuccess && progressive) e = cudaMallocHost((void**)&j->h_frame[1], std::max<size_t>(j->frame_bytes, 1));
    for (int k = 0; k < 2 && e == cudaSuccess; ++k) e = cudaEventCreateWithFlags(&j->ev_resolved[k], cudaEventDisableTiming);
    for (int k = 0; k < 2 && e == cudaSuccess; ++k) e = cudaEventCreateWithFlags(&j->pass_copied[k], cudaEventDisableTiming);
    j->band_copied.assign((size_t)j->n_bands, nullptr);
    for (int k = 0; k < j->n_bands && e == cudaSuccess && !progressive; ++k) e = cudaEventCreateWithFlags(&j->band_copied[k], cudaEventDisableTiming);
    if (e != cudaSuccess) {
        for (auto& h : j->h_frame) if (h) cudaFreeHost(h);
        for (auto& ev : j->ev_resolved) if (ev) cudaEventDestroy(ev);
        for (auto& ev : j->pass_copied) if (ev) cudaEventDestroy(ev);
        for (auto& ev : j->band_copied) if (ev) cudaEventDestroy(ev);
        delete j;
        return fail(RTB_ECUDA, std::string("rtb_job_begin: ") + cudaGetErrorString(e));
    }
    int n_workers = !progressive && j->n_bands >= 4 ? 2 : 1;
    if (const char* env = getenv("RTB_JOB_WORKERS")) n_workers = std::min(std::max(1, atoi(env)), std::max(1, j->n_bands));
    j->workers_running = n_workers;
    j->t_begin = std::chrono::steady_clock::now();
    for (int w = 0; w < n_workers; ++w) j->workers.emplace_back(job_worker, j, w);
    *out = j;
    return RTB_OK;
}

}  // namespace

extern "C" {

int rtb_job_begin(rtb_scene* scene, const rtb_params* params, int32_t passes, rtb_job** out) {
    return job_begin(scene, params, passes, nullptr, nullptr, out);
}

int rtb_job_begin_adaptive(rtb_scene* scene, const rtb_params* params, const rtb_adaptive* opts, rtb_job** out) {
    if (!scene || !out) return fail(RTB_EINVAL, "NULL argument");
    int rc = check_params(params);
    if (rc == RTB_OK) rc = check_adaptive(params, opts);
    if (rc != RTB_OK) return rc;
    return job_begin(scene, params, params->spp / opts->pass_spp, opts, nullptr, out);
}

int rtb_job_begin_denoised(rtb_scene* scene, const rtb_params* params, int32_t passes, const rtb_adaptive* adaptive,
                           const rtb_denoise* denoise, rtb_job** out) {
    if (!scene || !out) return fail(RTB_EINVAL, "NULL argument");
    int rc = check_params(params);
    if (rc == RTB_OK && adaptive) rc = check_adaptive(params, adaptive);
    if (rc == RTB_OK) rc = check_denoise(params, denoise);
    if (rc != RTB_OK) return rc;
    return job_begin(scene, params, adaptive ? params->spp / adaptive->pass_spp : passes, adaptive, denoise, out);
}

// returns 1 = record produced, 0 = frame(s) complete, RTB_ESTOPPED after a cancel, or another negative error
int rtb_job_next(rtb_job* job, uint16_t* x, uint16_t* y, uint8_t* n, uint8_t* rgb) {
    if (!job || !x || !y || !n || !rgb) return fail(RTB_EINVAL, "NULL argument");
    return job_next_record(job, true, x, y, n, rgb);
}

// whole-frame form of rtb_job_next: hands out the next finished pass in one copy (a single-pass job: the frame, once every band is in)
int rtb_job_next_frame(rtb_job* job, uint8_t* rgb8_out, int32_t* pass_index) {
    if (!job || !rgb8_out) return fail(RTB_EINVAL, "NULL argument");
    const int h = job->params.height;
    // a single-pass job delivers its frame once every band is in: walk the cursor to the last band
    for (;;) {
        const int rc = job_acquire_rows(job, true);
        if (rc != 1) return rc;
        if (job->avail_rows >= h) break;
        job->cursor_x = 0;
        job->cursor_y = job->avail_rows;
    }
    std::memcpy(rgb8_out, job->cur, job->frame_bytes);
    if (pass_index) *pass_index = job->pass_consumed;
    job_pass_consumed(job);
    return 1;
}

int rtb_job_next_messages(rtb_job* job, uint8_t* buf, int64_t buf_bytes, int32_t max_records, int64_t* bytes_written) {
    if (!job || !buf || !bytes_written) return fail(RTB_EINVAL, "NULL argument");
    int64_t off = 0;
    int produced = 0;
    while (produced < max_records && off + 6 + 3 * PIXELS_PER_MSG <= buf_bytes) {
        uint16_t x, y;
        uint8_t n;
        const int rc = job_next_record(job, produced == 0, &x, &y, &n, buf + off + 6);   // never block once something has been produced
        if (rc != 1) {
            *bytes_written = off;
            return produced > 0 ? produced : rc;
        }
        uint8_t* m = buf + off;  // header, src/server.rs:173-177
        m[0] = 0;
        m[1] = n;
        m[2] = (uint8_t)(x & 0xff); m[3] = (uint8_t)(x >> 8);
        m[4] = (uint8_t)(y & 0xff); m[5] = (uint8_t)(y >> 8);
        off += 6 + 3 * (int64_t)n;
        ++produced;
    }
    *bytes_written = off;
    return produced;
}

// counters of the job so far (finished bands / passes); first_record_ms and wall_ms are filled for jobs only
int rtb_job_stats(rtb_job* job, rtb_stats* stats) {
    if (!job || !stats) return fail(RTB_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(job->mu);
    *stats = job->stats;
    stats->first_record_ms = job->stats_first_ms.load();
    if (!job->finished) stats->wall_ms = ms_since(job->t_begin);
    return RTB_OK;
}

int rtb_job_cancel(rtb_job* job) {
    if (!job) return fail(RTB_EINVAL, "NULL job");
    std::lock_guard<std::mutex> lk(job->mu);
    job->cancel = 1;
    job->cv.notify_all();
    return RTB_OK;
}

int rtb_job_end(rtb_job* job) {
    if (!job) return fail(RTB_EINVAL, "NULL job");
    bool early;
    {
        std::lock_guard<std::mutex> lk(job->mu);
        early = !job->finished;
        if (early) job->cancel = 1;
        job->cv.notify_all();
    }
    for (auto& t : job->workers) if (t.joinable()) t.join();
    bool complete = job->passes > 1 ? job->passes_done >= job->passes || job->converged : true;
    for (char d : job->band_done) complete = complete && (job->passes > 1 || d);
    const int was_cancelled = job->cancel && job->error == RTB_OK && !complete;
    cudaSetDevice(job->scene->device);
    for (auto& h : job->h_frame) if (h) cudaFreeHost(h);
    for (auto& ev : job->ev_resolved) if (ev) cudaEventDestroy(ev);
    for (auto& ev : job->pass_copied) if (ev) cudaEventDestroy(ev);
    for (auto& ev : job->band_copied) if (ev) cudaEventDestroy(ev);
    delete job;
    return was_cancelled ? RTB_ECANCELLED : RTB_OK;
}

}  // extern "C"
