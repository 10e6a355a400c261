// wavefront.cuh — the wavefront path-tracing kernels (sm_100a).
//
// One iteration of the pipeline (all launches on one stream, every counter stays on the device):
//   k_prepare   1 thread: snapshot the free slots of the current path queue, reserve that many camera
//               samples, reset the other queue / the shadow queue / the work cursors
//   k_generate  primary-ray generation (sample_pixel's loop nest, src/server.rs:335-358)
//   k_traverse  Mesh::intersect for every ray that can reach the mesh box — the extension rays of this
//               iteration AND the shadow rays queued by the previous k_shade: persistent warps walk the LBVH
//               "while-while" and refill finished lanes with new rays, so the SIMD lanes stay busy although
//               incoherent rays need very different numbers of steps; unoccluded NEE candidates are added
//               to the fp32 sub-pixel accumulators here
//   k_shade     one level of Scene::reflected_radiance per path (src/scene.rs:161-244): emission, light
//               sample, russian roulette, BRDF sample.  It also runs the ANALYTIC half of Scene::trace_ray
//               (planes, spheres: the same short table for every lane, no divergence) for the two rays it
//               creates, so that only rays which still need the mesh are queued for a traversal kernel
//   k_resolve   sample_pixel's tail + gamma_correct + `as u8` (src/server.rs:360-368, 187-189)
// Queues are structure-of-arrays (float4 lanes, coalesced).  The path queue is two-ended: rays that need
// the BVH are appended from the front, rays whose analytic hit is already final from the back, with
// warp-aggregated atomics; k_extend only visits the front part.
#pragma once

#include "adaptive_rule.cuh"
#include "intersect.cuh"
#include "octree.cuh"
#include "shade.cuh"

namespace rtb {

constexpr int WF_THREADS = 256;
constexpr int TILE = 32;  // multi-GPU shard unit: 32x32 pixels, interleaved over ranks
constexpr uint32_t SHADOW_PROBE = 0x80000000u;  // shadow entry = dead-MIS probe resolved by a CLOSEST-hit query (mesh lights)
constexpr uint32_t MAX_DEPTH_FIELD = 4095u;
constexpr uint32_t FETCH_CHUNK = 32;     // ray indices a warp reserves per atomic
constexpr int REFILL_BELOW = 28;         // default: refill a warp when fewer than this many lanes are still traversing
#ifndef RTB_PARK_BELOW
#define RTB_PARK_BELOW 20
#endif
#ifndef RTB_SHADE_CHUNK
#define RTB_SHADE_CHUNK 64
#endif
constexpr uint32_t SHADE_CHUNK = RTB_SHADE_CHUNK;     // queue entries a k_shade warp reserves per atomic
constexpr int SHADE_PARK_BELOW = RTB_PARK_BELOW;      // k_shade tail: park the paths of a warp with fewer live lanes than this once the queue is drained
constexpr uint32_t SHADE_SEG = 128;      // OUTPUT slots a k_shade warp reserves per atomic in each queue class
constexpr uint32_t HIT_HOLE = 0xffffffffu;       // path-queue slot reserved by a k_shade warp but never filled (hit.y)
constexpr uint32_t TLIM_HOLE = 0xff800000u;      // same for the shadow queue (d.w = -inf)
constexpr int INNER_STEPS = 8;           // default: inner-node steps a lane may take before the warp re-checks for idle lanes

struct PathQueue {   // capacity P each
    float4* o;       // origin.xyz | pcode of the primitive the ray starts on (+ flags)
    float4* d;       // direction.xyz | accumulator index (pixel*4 + sub-pixel)
    float4* beta;    // throughput.rgb | (sample << 12 | depth of the vertex this ray will hit)
    float4* ov;      // stale `o` (only read when PC_STALE_O is set)
    float2* hit;     // nearest hit so far: t | id (analytic result at creation, refined by k_extend)
};

struct ShadowQueue {  // capacity SP
    float4* o;        // x.xyz | pcode
    float4* d;        // direction.xyz | tlimit (|y - x| - ERR_MARGIN; probes: analytic hit distance)
    float4* c;        // contribution.rgb | accumulator index (| SHADOW_PROBE)
};

// Every hot counter sits on its own 128-byte line: atomics to words of one line serialise in one L2 slice.
struct alignas(128) PaddedCounter {
    uint32_t v;
    uint32_t pad[31];
};
struct DevCtrl {
    PaddedCounter ext_head_[2], ext_tail_[2], sh_head_[2], cursor_trav_, cursor_shade_;
    uint32_t gen_count;
    int32_t tile_base, n_tiles;   // local tiles [tile_base, tile_base + n_tiles) are the frame region of this run (streaming jobs go band by band)
    uint32_t live[2], sh_live[2];   // FILLED entries of path / shadow queue c (the heads / tails also count reserved-but-unfilled slots)
    uint32_t active;        // paths alive in the current queue after k_prepare (+ reserved samples + pending shadow rays)
    unsigned long long gen_base, work_next, work_total;
    unsigned long long samples, rays_primary, rays_extension, rays_shadow, iterations;
    unsigned long long rays_bvh, shadow_bvh;   // of those, how many needed a BVH traversal
    unsigned long long paths_queued;           // path-queue entries written by k_shade
    uint32_t overflow;                         // queue slots refused because they lay beyond the physical capacity (must stay 0)
    unsigned long long node_visits, tri_tests;
    // counting build only: SIMD-slot accounting of k_traverse (lane-slots offered vs used)
    unsigned long long dbg[8];   // 0 rounds, 1 inner slot-steps offered (32 x trips), 2 leaf phases, 3 leaf lanes, 4 refills, 5 refilled lanes, 6 rays, 7 -
};
#define ext_head(i) ext_head_[i].v
#define ext_tail(i) ext_tail_[i].v
#define sh_head(i) sh_head_[i].v
#define cursor_trav cursor_trav_.v
#define cursor_shade cursor_shade_.v

struct RenderArgs {
    DevScene S;
    Camera cam;
    int width, height, spp, num_samples;
    uint32_t ks_done;    // samples resolved so far, in (k*4 + sub-pixel) units; 4*num_samples for a finished frame
    PhiloxKeys keys;     // round keys of the frame's seed
    SmallScene ss;       // analytic table of small scenes (k_shade<MODE, NP, NS> with NP > 0)
    int estimator;
    int rank, world, tiles_x, tiles_y, n_local_tiles;
    int tile_base;       // first LOCAL tile of this launch series (streaming jobs render a frame band by band; 0 = whole shard)
    const int32_t* tile_list;   // adaptive passes (world = 1): k_generate's local tile lt is tile tile_list[lt]; nullptr = lt + tile_base
    const uint32_t* tile_ks;    // adaptive resolve: ks_done per tile (indexed by tile); nullptr = ks_done for every tile
    uint32_t P, SP;          // most paths / shadow rays alive at once
    uint32_t Pcap, SPcap;    // physical slots per queue: P, SP + room for the unfilled tails of k_shade's per-warp segments
    PathQueue q[2];
    // the queues of THIS launch, resolved on the host (q[c], q[1 - c], sq[c], sq[1 - c]): plain constant-bank pointers
    // instead of parameter arrays indexed by a run-time `c`
    PathQueue qin, qout;
    ShadowQueue sqin, sqout;
    float4 light_sphere;     // centre | radius of a sphere light
    float light_pdf;         // 1 / (4 pi r^2)
    ShadowQueue sq[2];   // sq[c] is read by k_traverse(c) and was written by k_shade(1-c)
    float4* accum;       // [pixel*4 + sub] -> (r, g, b, -) sums
    DevCtrl* ctrl;
    // probe mode (rtb_sample_radiance): explicit work items, accumulator index = item index
    const int32_t* probe_px;
    const int32_t* probe_py;
    const int32_t* probe_sample;
    int n_probe;
    int pixel_list;      // 1: probe_px / probe_py list PIXELS (rtb_sample_pixels): every listed pixel gets the full sample set,
                         //    work order (k, sub-pixel) major like a frame, accumulator index = list index * 4 + sub-pixel
    int tune_refill, tune_steps;   // traversal knobs (0 = defaults above); rtb_params.reserved[1], [2]
    // graph mode (small frames): k_prepare publishes {iteration, live paths} to mapped pinned host memory so the
    // host can stop launching without a copy or an event per iteration
    volatile unsigned long long* host_state;
    uint32_t trav_warps;   // warps in the k_traverse grid: each owns the static first chunk [w*32, w*32+32)
    uint32_t shade_warps;  // same for k_shade
    // coherence binning of the LBVH rays (k_bin_*): perm[i] = queue index of the i-th ray in bin order; nullptr = queue order
    uint32_t* bin_key;     // [Pcap + SPcap]
    uint32_t* bin_perm;    // [Pcap + SPcap]
    uint32_t* bin_hist;    // [BIN_MAX + 1], zero between iterations
    uint32_t* bin_offs;    // [BIN_MAX + 1]
    int bin_bits;          // cell bits per axis (0 = binning off); bins = 8 octants x 2^(3 bits)
    int bin_octant_major;
    int accel;             // RTB_ACCEL_*: 1 = the mesh rays go through the reference's octrees (k_traverse_octree)
};

// ---------------------------------------------------------------- tile order <-> pixels
// local pixel index lp = local_tile * 1024 + slot; slot walks 8x4 pixel blocks (one warp each).
__host__ __device__ __forceinline__ bool local_to_xy(int lp, int rank, int world, int tiles_x, int width, int height, int& x, int& y) {
    int lt = lp >> 10, slot = lp & 1023;
    int t = lt * world + rank;
    int ty = t / tiles_x, tx = t - ty * tiles_x;
    int blk = slot >> 5, lane = slot & 31;
    x = tx * TILE + (blk & 3) * 8 + (lane & 7);
    y = ty * TILE + (blk >> 2) * 4 + (lane >> 3);
    return x < width && y < height;
}

// ---------------------------------------------------------------- warp-aggregated queue pushes
// All 32 lanes call these.  One lane issues the (independent) atomics back to back, so their latencies overlap.
struct PushSlots {
    uint32_t ext, sh, pr;
};
__device__ __forceinline__ PushSlots push_all(uint32_t* ext_head, uint32_t* ext_tail, uint32_t* sh_head, bool ext_push,
                                              bool ext_front, bool sh_push, bool pr_push) {
    const unsigned lane = threadIdx.x & 31;
    const unsigned mf = __ballot_sync(0xffffffffu, ext_push && ext_front);
    const unsigned mb = __ballot_sync(0xffffffffu, ext_push && !ext_front);
    const unsigned ms = __ballot_sync(0xffffffffu, sh_push);
    const unsigned mp = __ballot_sync(0xffffffffu, pr_push);
    uint32_t bf = 0, bb = 0, bs = 0;
    if (lane == 0) {
        if (mf) bf = atomicAdd(ext_head, (uint32_t)__popc(mf));
        if (mb) bb = atomicSub(ext_tail, (uint32_t)__popc(mb));
        if (ms | mp) bs = atomicAdd(sh_head, (uint32_t)(__popc(ms) + __popc(mp)));
    }
    bf = __shfl_sync(0xffffffffu, bf, 0);
    bb = __shfl_sync(0xffffffffu, bb, 0);
    bs = __shfl_sync(0xffffffffu, bs, 0);
    const unsigned below = (1u << lane) - 1u;
    PushSlots r;
    r.ext = ext_front ? bf + __popc(mf & below) : bb - 1u - __popc(mb & below);
    r.sh = bs + __popc(ms & below);
    r.pr = bs + __popc(ms) + __popc(mp & below);
    return r;
}

#ifndef RTB_SHADE_THREADS
#define RTB_SHADE_THREADS 256
#endif
#ifndef RTB_SHADE_MINB
#define RTB_SHADE_MINB (512 / RTB_SHADE_THREADS)
#endif
constexpr int SHADE_THREADS = RTB_SHADE_THREADS;   // CTA size of k_shade (warps are independent: only occupancy depends on it)

__device__ __forceinline__ void accum_add(float4* accum, uint32_t idx, float3 v) {
    atomicAdd(&accum[idx], make_float4(v.x, v.y, v.z, 0.0f));  // one 128-bit RED (sm_90+)
}

__device__ __forceinline__ int object_of(const DevScene& S, const SharedScene& sh, uint32_t id) {
    if (id < TRI_BASE) return sh.prims[id].obj;
    return __float_as_int(__ldg(S.tri_nrm + (id - TRI_BASE)).w);
}

// ---------------------------------------------------------------- k_prepare
__global__ void k_prepare(RenderArgs a, int c) {
    DevCtrl* C = a.ctrl;
    const uint32_t live = C->live[c];           // paths k_shade(1 - c) handed on
    const uint32_t free_slots = a.P - live;
    unsigned long long remaining = C->work_total - C->work_next;
    uint32_t n_new = remaining < (unsigned long long)free_slots ? (uint32_t)remaining : free_slots;
    C->gen_base = C->work_next;
    C->gen_count = n_new;
    C->work_next += n_new;
    C->ext_head(1 - c) = 0;
    C->ext_tail(1 - c) = a.Pcap;
    C->sh_head(1 - c) = 0;
    C->live[1 - c] = 0;
    C->sh_live[1 - c] = 0;
    C->cursor_trav = a.trav_warps * FETCH_CHUNK;   // chunks below that are handed out statically (no atomic)
    C->cursor_shade = a.shade_warps * SHADE_CHUNK;
    C->active = live + n_new + C->sh_live[c];   // pending shadow rays keep the loop alive
    C->iterations++;
    if (a.host_state) {
        a.host_state[1] = C->active;
        __threadfence_system();
        a.host_state[0] = C->iterations;
    }
}

// ---------------------------------------------------------------- k_generate
template <int NP = 0, int NS = 0>
__global__ void __launch_bounds__(WF_THREADS) k_generate(const __grid_constant__ RenderArgs a, int c) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DevCtrl* C = a.ctrl;
    const uint32_t n = C->gen_count;
    if (blockIdx.x * WF_THREADS >= n) return;   // tail iterations: most CTAs have nothing to generate
    const SharedScene sh = stage_scene(a.S, smem_raw, false);
    const unsigned long long base = C->gen_base;
    const unsigned lane = threadIdx.x & 31;
    const uint32_t nwarps_total = (gridDim.x * blockDim.x) >> 5;
    const uint32_t warp_id = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const float w = (float)a.width, h = (float)a.height;
    uint32_t made = 0, made_bvh = 0;
    for (uint32_t b = warp_id * 32; b < n; b += nwarps_total * 32) {
        uint32_t j = b + lane;
        bool valid = j < n;
        float4 o4 = make_float4(0, 0, 0, 0), d4 = o4, b4 = o4;
        float2 h2 = make_float2(0.f, 0.f);
        bool front = false;
        if (valid) {
            unsigned long long wi = base + j;
            int x, y, sample;
            uint32_t acc, rng_pixel;
            if (a.probe_px && !a.pixel_list) {
                x = a.probe_px[wi];
                y = a.probe_py[wi];
                sample = a.probe_sample[wi];
                acc = (uint32_t)wi;
                rng_pixel = (uint32_t)(y * a.width + x);
            } else {
                // work order: (k, sub-pixel) major, local pixel minor -> neighbouring lanes = neighbouring pixels
                unsigned long long npl = a.pixel_list ? (unsigned long long)a.n_probe : (unsigned long long)C->n_tiles * 1024ull;
                uint32_t ks = (uint32_t)(wi / npl);
                int lp = (int)(wi - (unsigned long long)ks * npl);
                int k = ks >> 2, sub = ks & 3;
                if (a.pixel_list) {
                    x = a.probe_px[lp];
                    y = a.probe_py[lp];
                    acc = (uint32_t)lp * 4u + (uint32_t)sub;
                } else {
                    const int lt = lp >> 10;
                    const int t = a.tile_list ? a.tile_list[lt] : lt + C->tile_base;
                    valid = local_to_xy(t * 1024 + (lp & 1023), a.rank, a.world, a.tiles_x, a.width, a.height, x, y);
                    acc = (uint32_t)(y * a.width + x) * 4u + (uint32_t)sub;
                }
                sample = sub * a.num_samples + k;
                rng_pixel = (uint32_t)(y * a.width + x);
            }
            if (valid) {
                int sub = sample / a.num_samples;
                float4 r = rng_block(rng_pixel, (uint32_t)sample, 0u, 0u, a.keys);
                float3 dir = camera_dir(a.cam, x, a.height - y - 1, sub & 1, sub >> 1, tent(r.x), tent(r.y), w, h);
                float ta;
                uint32_t ida;
                if (NP > 0) analytic_closest_small<NP, NS>(a.ss, -1, a.cam.pos, dir, PC_NONE, ta, ida);
                else analytic_closest(sh, a.S.n_planes, a.S.n_prims, a.cam.pos, dir, PC_NONE, ta, ida);
                front = ray_hits_bvh_box(a.S, a.cam.pos, dir, ta);
                o4 = make_float4(a.cam.pos.x, a.cam.pos.y, a.cam.pos.z, __uint_as_float(PC_NONE));
                d4 = make_float4(dir.x, dir.y, dir.z, __uint_as_float(acc));
                b4 = make_float4(1.f, 1.f, 1.f, __uint_as_float(((uint32_t)sample << 12) | 1u));
                h2 = make_float2(ta, __uint_as_float(ida));
            }
        }
        PushSlots ps = push_all(&C->ext_head(c), &C->ext_tail(c), &C->sh_head(c), valid, front, false, false);
        if (valid && ps.ext >= a.Pcap) { atomicAdd(&C->overflow, 1u); valid = false; }
        if (valid) {
            a.qin.o[ps.ext] = o4;
            a.qin.d[ps.ext] = d4;
            a.qin.beta[ps.ext] = b4;
            a.qin.hit[ps.ext] = h2;
            ++made;
            made_bvh += front ? 1u : 0u;
        }
    }
    for (int off = 16; off; off >>= 1) {
        made += __shfl_down_sync(0xffffffffu, made, off);
        made_bvh += __shfl_down_sync(0xffffffffu, made_bvh, off);
    }
    if (lane == 0 && made) {
        atomicAdd(&C->samples, (unsigned long long)made);
        atomicAdd(&C->rays_primary, (unsigned long long)made);
        if (made_bvh) atomicAdd(&C->rays_bvh, (unsigned long long)made_bvh);
    }
}

// ---------------------------------------------------------------- coherence binning of the LBVH rays
// k_traverse's warps lose half their lanes to divergence when the 32 rays of a warp walk unrelated parts of the tree
// (incoherent bounce rays in queue order).  Before each traversal the rays of the iteration — the front class of the
// path queue and the queued shadow rays — are therefore BINNED by (cell of the point where the ray enters the mesh
// box | direction octant) with a one-pass counting sort: keys + histogram, exclusive scan, scatter of the INDICES.
// k_traverse fetches its rays through the permutation; nothing else moves.  All counts stay on the device.
constexpr int BIN_MAX_BITS = 5;                                  // cell bits per axis
constexpr uint32_t BIN_MAX = 8u << (3 * BIN_MAX_BITS);           // bins at BIN_MAX_BITS (holes go to bin index `bins`)
constexpr int BIN_SCAN_THREADS = 1024;

__device__ __forceinline__ uint32_t spread3_5(uint32_t v) {   // bit k of a 5-bit value -> bit 3k
    return (v & 1u) | ((v & 2u) << 2) | ((v & 4u) << 4) | ((v & 8u) << 6) | ((v & 16u) << 8);
}
__device__ __forceinline__ uint32_t bin_key_of(const RenderArgs& a, float3 o, float3 d) {
    // entry point into the box of all triangles (the origin itself when it lies inside)
    auto inv = [](float v) { return fast_rcp(fabsf(v) > 1e-20f ? v : copysignf(1e-20f, v)); };
    const float ix = inv(d.x), iy = inv(d.y), iz = inv(d.z);
    const float x0 = (a.S.bvh_min.x - o.x) * ix, x1 = (a.S.bvh_max.x - o.x) * ix;
    const float y0 = (a.S.bvh_min.y - o.y) * iy, y1 = (a.S.bvh_max.y - o.y) * iy;
    const float z0 = (a.S.bvh_min.z - o.z) * iz, z1 = (a.S.bvh_max.z - o.z) * iz;
    const float tmin = fmaxf(fmaxf(fminf(x0, x1), fminf(y0, y1)), fmaxf(fminf(z0, z1), 0.0f));
    const float3 p = o + tmin * d;
    const float cells = (float)(1 << a.bin_bits);
    const float3 e = a.S.bvh_max - a.S.bvh_min;
    const int hi = (1 << a.bin_bits) - 1;
    const int cx = min(max((int)((p.x - a.S.bvh_min.x) * cells * fast_rcp(fmaxf(e.x, 1e-20f))), 0), hi);
    const int cy = min(max((int)((p.y - a.S.bvh_min.y) * cells * fast_rcp(fmaxf(e.y, 1e-20f))), 0), hi);
    const int cz = min(max((int)((p.z - a.S.bvh_min.z) * cells * fast_rcp(fmaxf(e.z, 1e-20f))), 0), hi);
    const uint32_t morton = spread3_5((uint32_t)cx) | (spread3_5((uint32_t)cy) << 1) | (spread3_5((uint32_t)cz) << 2);
    const uint32_t oct = (d.x < 0.f ? 1u : 0u) | (d.y < 0.f ? 2u : 0u) | (d.z < 0.f ? 4u : 0u);
    return a.bin_octant_major ? (oct << (3 * a.bin_bits)) | morton : (morton << 3) | oct;
}

__global__ void __launch_bounds__(WF_THREADS) k_bin_keys(const __grid_constant__ RenderArgs a, int c) {
    DevCtrl* C = a.ctrl;
    const uint32_t n_ext = min(C->ext_head(c), a.Pcap);   // (the heads also count slots refused for lack of capacity — an error the host reports)
    const uint32_t count = n_ext + min(C->sh_head(c), a.SPcap);
    const uint32_t bins = 8u << (3 * a.bin_bits);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x) {
        float4 o4, d4;
        bool hole;
        if (i < n_ext) {
            hole = __float_as_uint(a.qin.hit[i].y) == HIT_HOLE;
            o4 = a.qin.o[i];
            d4 = a.qin.d[i];
        } else {
            d4 = a.sqin.d[i - n_ext];
            hole = __float_as_uint(d4.w) == TLIM_HOLE;
            o4 = a.sqin.o[i - n_ext];
        }
        const uint32_t key = hole ? bins : bin_key_of(a, f3(o4), f3(d4));   // unfilled slots sort to the end
        a.bin_key[i] = key;
        atomicAdd(&a.bin_hist[key], 1u);
    }
}

// one CTA: exclusive scan of the histogram into the scatter offsets; clears the histogram for the next iteration
__global__ void __launch_bounds__(BIN_SCAN_THREADS) k_bin_scan(const __grid_constant__ RenderArgs a) {
    __shared__ uint32_t warp_sum[BIN_SCAN_THREADS / 32];
    const uint32_t n = (8u << (3 * a.bin_bits)) + 1u;
    const uint32_t per = (n + BIN_SCAN_THREADS - 1) / BIN_SCAN_THREADS;
    const uint32_t b0 = min(threadIdx.x * per, n), b1 = min(b0 + per, n);
    uint32_t sum = 0;
    for (uint32_t b = b0; b < b1; ++b) sum += a.bin_hist[b];
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t incl = sum;
    for (int off = 1; off < 32; off <<= 1) {
        const uint32_t v = __shfl_up_sync(0xffffffffu, incl, off);
        if ((int)lane >= off) incl += v;
    }
    if (lane == 31) warp_sum[w] = incl;
    __syncthreads();
    if (w == 0) {
        uint32_t v = warp_sum[lane];
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t u = __shfl_up_sync(0xffffffffu, v, off);
            if ((int)lane >= off) v += u;
        }
        warp_sum[lane] = v;   // inclusive over warps
    }
    __syncthreads();
    uint32_t run = incl - sum + (w ? warp_sum[w - 1] : 0u);
    for (uint32_t b = b0; b < b1; ++b) {
        const uint32_t h = a.bin_hist[b];
        a.bin_offs[b] = run;
        a.bin_hist[b] = 0u;
        run += h;
    }
}

__global__ void __launch_bounds__(WF_THREADS) k_bin_scatter(const __grid_constant__ RenderArgs a, int c) {
    DevCtrl* C = a.ctrl;
    const uint32_t count = min(C->ext_head(c), a.Pcap) + min(C->sh_head(c), a.SPcap);
    for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x)
        a.bin_perm[atomicAdd(&a.bin_offs[a.bin_key[i]], 1u)] = i;
}

// ---------------------------------------------------------------- persistent traversal kernels
// Warp-level work fetch: a warp owns [wnext, wend) of the queue and takes a new FETCH_CHUNK with one
// atomic when it runs dry.  Returns false once the queue is exhausted.  Warp-uniform.
__device__ __forceinline__ bool warp_reserve(uint32_t* cursor, uint32_t count, uint32_t& wnext, uint32_t& wend) {
    if (wnext < wend) return true;
    uint32_t b = 0;
    if ((threadIdx.x & 31) == 0) b = atomicAdd(cursor, FETCH_CHUNK);
    b = __shfl_sync(0xffffffffu, b, 0);
    if (b >= count) return false;
    wnext = b;
    wend = min(b + FETCH_CHUNK, count);
    return true;
}

// k_traverse: every LBVH query of one iteration in ONE persistent launch —
//   * closest hit for the front (BVH) class of path queue c            (Mesh::intersect; updates q.hit in place)
//   * any hit for the NEE candidates in shadow queue c                  (mutually_visible; accumulates if unoccluded)
//   * closest hit for dead-MIS probes against a mesh light              (hit.id == light_source test)
// Lanes refill individually from one work cursor, so the two ray kinds share warps and the tail is paid once.
template <bool COUNT, int MINB = 4, bool WIDE = false>
__global__ void __launch_bounds__(WF_THREADS, MINB) k_traverse(const __grid_constant__ RenderArgs a, int c) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(reinterpret_cast<int*>(smem_raw) + threadIdx.x), sstride = blockDim.x * 4u;
    int lstack[STACK_LOCAL];
    DevCtrl* C = a.ctrl;
    const uint32_t n_ext = min(C->ext_head(c), a.Pcap);   // only the BVH class of the path queue needs a traversal
    const uint32_t count = n_ext + min(C->sh_head(c), a.SPcap);
    const unsigned lane = threadIdx.x & 31;
    const PathQueue& Q = a.qin;
    const ShadowQueue& SQ = a.sqin;
    const int light_obj = a.S.hdr->light_obj;
    const uint32_t* const perm = a.bin_bits > 0 ? a.bin_perm : nullptr;   // bin order (see k_bin_*), or queue order
    const int refill_below = a.tune_refill > 0 ? a.tune_refill : REFILL_BELOW;
    const int steps = a.tune_steps > 0 ? a.tune_steps : (WIDE ? INNER_STEPS / 2 : INNER_STEPS);
    uint32_t work[2] = {0, 0};
    unsigned long long dbg[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // first chunk: static (warp w owns [w*32, w*32+32)), later chunks from the atomic cursor, which k_prepare
    // starts behind the static region — a launch with few rays does no atomics at all
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t wnext = min(gwarp * FETCH_CHUNK, count), wend = min(gwarp * FETCH_CHUNK + FETCH_CHUNK, count);
    bool exhausted = false;
    if (blockIdx.x * (WF_THREADS / 32) * FETCH_CHUNK >= count) return;   // whole CTA beyond the static region of a small launch
    Trav T;
    T.node = NODE_SENTINEL;
    T.sp = 0;
    T.best_id = PC_NONE;
    T.tlimit = 0.f;
    uint32_t slot = 0;
    int kind = -1;            // -1 none, 0 extension (closest), 1 shadow (any hit), 2 probe (closest, mesh light)
    bool occluded = false;

    for (;;) {
        // ---- retire finished rays
        const bool idle = T.node == NODE_SENTINEL;
        if (idle && kind >= 0) {
            if (kind == 0) {
                if (T.best_id != PC_NONE) Q.hit[slot] = make_float2(T.tlimit, __uint_as_float(T.best_id));
            } else {
                bool add;
                if (kind == 2) add = T.best_id != PC_NONE && __float_as_int(__ldg(a.S.tris + (size_t)(T.best_id - TRI_BASE) * TRI_STRIDE + 2).w) == light_obj;
                else add = !occluded;
                if (add) {
                    const float4 c4 = SQ.c[slot];
                    accum_add(a.accum, __float_as_uint(c4.w) & ~SHADOW_PROBE, f3(c4));
                }
            }
            kind = -1;
        }
        // ---- refill idle lanes
        const unsigned idle_mask = __ballot_sync(0xffffffffu, idle);
        if (idle_mask && !exhausted) {
            if (!warp_reserve(&C->cursor_trav, count, wnext, wend)) exhausted = true;
            else {
                const uint32_t pos = wnext + __popc(idle_mask & ((1u << lane) - 1u));
                if (idle && pos < wend) {
                    const uint32_t my = perm ? perm[pos] : pos;
                    // slots a k_shade warp reserved but did not fill are marked as holes: the lane stays idle this round
                    if (my < n_ext) {
                        const float2 h2 = Q.hit[my];
                        if (__float_as_uint(h2.y) != HIT_HOLE) {
                            slot = my;
                            kind = 0;
                            const float4 o4 = Q.o[my], d4 = Q.d[my];
                            trav_begin(a.S, T, f3(o4), f3(d4), __float_as_uint(o4.w), h2.x, WIDE ? a.S.root4 : a.S.root);
                        }
                    } else {
                        const float4 d4 = SQ.d[my - n_ext];
                        if (__float_as_uint(d4.w) != TLIM_HOLE) {
                            slot = my - n_ext;
                            const float4 o4 = SQ.o[slot];
                            kind = (__float_as_uint(SQ.c[slot].w) & SHADOW_PROBE) ? 2 : 1;
                            occluded = false;
                            trav_begin(a.S, T, f3(o4), f3(d4), __float_as_uint(o4.w), d4.w, WIDE ? a.S.root4 : a.S.root);
                        }
                    }
                }
                if (COUNT && lane == 0) { dbg[4] += 1; dbg[5] += min((uint32_t)__popc(idle_mask), wend - wnext); }
                wnext = min(wnext + (uint32_t)__popc(idle_mask), wend);
            }
        }
        const unsigned active = __ballot_sync(0xffffffffu, T.node != NODE_SENTINEL);
        if (active == 0) {
            if (exhausted) break;
            continue;
        }
        // ---- traverse until too few lanes are left (then go back and refill).  A lane takes at most
        // `steps` inner nodes per round, so lanes whose ray ended are not left idle behind one long descent.
        for (;;) {
            int trips = 0;
            if (!COUNT && !WIDE && steps == INNER_STEPS) {   // default knob: unrolled, no loop counter
#pragma unroll
                for (int k = 0; k < INNER_STEPS; ++k) {
                    if (T.node < 0) break;
                    trav_inner<COUNT>(a.S, T, sbase, sstride, lstack, work);
                }
            } else {
                for (int k = 0; k < steps && T.node >= 0; ++k) {
                    if (WIDE) trav_inner4<COUNT>(a.S, T, sbase, sstride, lstack, work);
                    else trav_inner<COUNT>(a.S, T, sbase, sstride, lstack, work);
                    ++trips;
                }
            }
            if (COUNT) {
                int mx = trips;
                for (int off = 16; off; off >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, off));
                const unsigned lm = __ballot_sync(0xffffffffu, T.node < 0 && T.node != NODE_SENTINEL);
                if (lane == 0) { dbg[0] += 1; dbg[1] += 32ull * mx; dbg[2] += lm ? 1 : 0; dbg[3] += __popc(lm); }
            }
            if (T.node < 0 && T.node != NODE_SENTINEL) {
                // one instance of the leaf code for all ray kinds (shadow rays share warps with extension rays): an
                // any-hit query is a closest-hit query that stops after the first leaf with a hit below its limit
                trav_leaf<false, COUNT>(a.S, T, work);
                if (kind == 1 && T.best_id != PC_NONE) {
                    occluded = true;
                    T.node = NODE_SENTINEL;
                } else {
                    trav_pop(T, sbase, sstride, lstack);
                }
            }
            const unsigned act = __ballot_sync(0xffffffffu, T.node != NODE_SENTINEL);
            if (act == 0 || (!exhausted && __popc(act) < refill_below)) break;
        }
    }
    if (COUNT) {
        for (int off = 16; off; off >>= 1) {
            work[0] += __shfl_down_sync(0xffffffffu, work[0], off);
            work[1] += __shfl_down_sync(0xffffffffu, work[1], off);
        }
        if (lane == 0) {
            atomicAdd(&C->node_visits, (unsigned long long)work[0]);
            atomicAdd(&C->tri_tests, (unsigned long long)work[1]);
            for (int k = 0; k < 6; ++k) atomicAdd(&C->dbg[k], dbg[k]);
        }
    }
}

// k_traverse_octree: the same job as k_traverse — every mesh query of one iteration — under RTB_ACCEL_OCTREE_REFERENCE:
// each ray walks the reference's octrees (octree.cuh) instead of the LBVH.  One ray per thread, grid-stride; the octree
// search is not a nearest-hit query, so a shadow ray cannot stop at the first triangle below its limit either: it takes
// the hit the reference's trace_ray would see and compares (mutually_visible, src/scene.rs:258-270).
// Persistent, like k_traverse: a lane that has finished its ray takes the next one while its neighbours are still searching,
// and the search itself is cut into uniform steps — ONE child-box test per lane and step (oct_step), leaves tested in a phase
// of their own — so that lanes at different depths of different octrees still execute the same instruction.  (The first
// version ran oct_trace_meshes once per thread: ncu counted 5.8 of 32 lanes active per instruction.)
enum : int { OCT_IDLE = 0, OCT_NEXT_MESH, OCT_DESCEND, OCT_LEAF, OCT_DONE };
constexpr int OCT_STEPS = 12;   // child-box tests per lane and round (swept 6 .. 24 with refill thresholds 24 / 28: flat between 8 and 12)

template <bool COUNT>
__global__ void __launch_bounds__(WF_THREADS, 4) k_traverse_octree(const __grid_constant__ RenderArgs a, int c) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int2* const nstack = reinterpret_cast<int2*>(smem_raw) + threadIdx.x;   // (first child, mask) of the parent at level l: nstack[l * blockDim.x]
    const unsigned nstride = blockDim.x;
    DevCtrl* C = a.ctrl;
    const uint32_t n_ext = min(C->ext_head(c), a.Pcap);
    const uint32_t count = n_ext + min(C->sh_head(c), a.SPcap);
    const unsigned lane = threadIdx.x & 31;
    const int light_obj = a.S.hdr->light_obj;
    const uint32_t* const perm = a.bin_bits > 0 ? a.bin_perm : nullptr;   // bin order: neighbouring lanes walk neighbouring octants
    const int refill_below = a.tune_refill > 0 ? a.tune_refill : REFILL_BELOW;
    const int steps = a.tune_steps > 0 ? a.tune_steps : OCT_STEPS;
    const float4* const N = a.S.oct_nodes;
    uint32_t work[2] = {0, 0};
    const uint32_t gwarp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    uint32_t wnext = min(gwarp * FETCH_CHUNK, count), wend = min(gwarp * FETCH_CHUNK + FETCH_CHUNK, count);
    bool exhausted = false;
    if (blockIdx.x * (WF_THREADS / 32) * FETCH_CHUNK >= count) return;
    // lane state: the ray, the best hit so far over the analytic primitives and the meshes already searched, the search position
    float3 o = f3(0.f, 0.f, 0.f), d = o, inv = o;
    uint32_t origin = 0, best_id = PC_NONE, slot = 0, order = 0;
    float best_t = 0.f;
    uint2 obytes = make_uint2(0u, 0u);   // per octant one byte: 1 << its position in `order` (oct_order_bytes)
    uint32_t rem = 0;                  // see phase (2)
    int level = 0, mesh = -1, leaf_first = 0, leaf_cnt = 0;
    int cur_base = 0, cur_mask = 0;    // the parent being searched: its first child and which octants have one
    int phase = OCT_IDLE, kind = -1;   // kind: 0 extension, 1 NEE shadow ray, 2 dead-MIS probe

    for (;;) {
        // ---- retire finished rays
        if (phase == OCT_DONE) {
            if (kind == 0) {
                if (best_id != PC_NONE) a.qin.hit[slot] = make_float2(best_t, __uint_as_float(best_id));
            } else {
                const float4 c4 = a.sqin.c[slot];
                bool add;
                if (kind == 2) add = best_id != PC_NONE && __float_as_int(__ldg(a.S.tris + (size_t)(best_id - TRI_BASE) * TRI_STRIDE + 2).w) == light_obj;
                else add = best_id == PC_NONE;   // no mesh hit below the limit: visible
                if (add) accum_add(a.accum, __float_as_uint(c4.w) & ~SHADOW_PROBE, f3(c4));
            }
            phase = OCT_IDLE;
            kind = -1;
        }
        // ---- refill idle lanes
        const unsigned idle_mask = __ballot_sync(0xffffffffu, phase == OCT_IDLE);
        if (idle_mask && !exhausted) {
            if (!warp_reserve(&C->cursor_trav, count, wnext, wend)) exhausted = true;
            else {
                const uint32_t q = wnext + __popc(idle_mask & ((1u << lane) - 1u));
                if (phase == OCT_IDLE && q < wend) {
                    const uint32_t my = perm ? perm[q] : q;
                    float4 o4, d4;
                    bool take = false;
                    if (my < n_ext) {
                        const float2 h2 = a.qin.hit[my];
                        if (__float_as_uint(h2.y) != HIT_HOLE) {
                            take = true;
                            slot = my;
                            kind = 0;
                            o4 = a.qin.o[my];
                            d4 = a.qin.d[my];
                            best_t = h2.x;
                        }
                    } else {
                        d4 = a.sqin.d[my - n_ext];
                        if (__float_as_uint(d4.w) != TLIM_HOLE) {
                            take = true;
                            slot = my - n_ext;
                            o4 = a.sqin.o[slot];
                            kind = (__float_as_uint(a.sqin.c[slot].w) & SHADOW_PROBE) ? 2 : 1;
                            best_t = d4.w;   // NEE candidate: |y - x| - margin; dead-MIS probe: the analytic hit distance
                        }
                    }
                    if (take) {
                        o = f3(o4);
                        d = f3(d4);
                        inv = f3(1.0f / d.x, 1.0f / d.y, 1.0f / d.z);
                        origin = __float_as_uint(o4.w);
                        best_id = PC_NONE;
                        mesh = -1;
                        phase = OCT_NEXT_MESH;
                    }
                }
                wnext = min(wnext + (uint32_t)__popc(idle_mask), wend);
            }
        }
        if (__ballot_sync(0xffffffffu, phase != OCT_IDLE) == 0) {
            if (exhausted) break;
            continue;
        }
        for (;;) {
            // ---- (1) Scene::trace_ray's loop over the objects (src/scene.rs:277-284): the next mesh, its root, its search order
            if (phase == OCT_NEXT_MESH) {
                int root = -1;
                // a NEE shadow ray is decided by the first mesh hit below its limit (visible iff none): the other meshes cannot change that
                if (!(kind == 1 && best_id != PC_NONE))
                    while (++mesh < a.S.n_oct_meshes && (root = __ldg(a.S.oct_roots + mesh)) < 0) {}
                if (root < 0) phase = OCT_DONE;
                else {
                    const float4 rmn = __ldg(N + (size_t)root * 2), rmx = __ldg(N + (size_t)root * 2 + 1);
                    if (__float_as_int(rmx.w) >= 0) {   // the root is a leaf (a mesh of at most SMALL_NODE triangles)
                        leaf_first = __float_as_int(rmn.w);
                        leaf_cnt = __float_as_int(rmx.w);
                        level = -1;
                        phase = OCT_LEAF;
                    } else {
                        order = oct_search_order(rmn, rmx, o);
                        obytes = oct_order_bytes(order);
                        level = 0;
                        cur_base = __float_as_int(rmn.w);
                        cur_mask = -1 - __float_as_int(rmx.w);
                        rem = oct_present_in_order(cur_mask, obytes);
                        phase = OCT_DESCEND;
                    }
                }
            }
            // ---- (2) child-box tests, at most `steps` per lane and round.  `rem` = the children of the current parent that are still
            // to be tried, as bits in SEARCH order (bit p = the p-th octant of `order` has a child): a step takes the lowest one, so
            // octants without a child (a third of all slots) never cost a step
            for (int k = 0; k < steps; ++k) {
                if (!__any_sync(0xffffffffu, phase == OCT_DESCEND)) break;
                if (phase != OCT_DESCEND) continue;
                if (rem == 0u) {   // this parent is exhausted without a hit
                    if (level == 0) phase = OCT_NEXT_MESH;
                    else {
                        --level;
                        const int2 up = nstack[level * nstride];
                        cur_base = up.x;
                        cur_mask = up.y & 255;
                        rem = (unsigned)up.y >> 8;
                    }
                    continue;
                }
                const unsigned p = (unsigned)__ffs((int)rem) - 1u;
                rem &= rem - 1u;
                const int i = (int)(order >> (3 * p)) & 7;
                const int ch = cur_base + __popc((unsigned)cur_mask & ((1u << i) - 1u));
                const float4 cmn = __ldg(N + (size_t)ch * 2), cmx = __ldg(N + (size_t)ch * 2 + 1);
                if (COUNT) work[0]++;
                if (!oct_box_hit(cmn, cmx, o, d, inv)) continue;
                const int cnt = __float_as_int(cmx.w);
                if (cnt >= 0) {   // leaf: tested in phase (3)
                    leaf_first = __float_as_int(cmn.w);
                    leaf_cnt = cnt;
                    phase = OCT_LEAF;
                } else if (level + 1 < OCT_MAX_DEPTH) {
                    nstack[level * nstride] = make_int2(cur_base, cur_mask | (int)(rem << 8));
                    ++level;
                    cur_base = __float_as_int(cmn.w);
                    cur_mask = -1 - cnt;
                    rem = oct_present_in_order(cur_mask, obytes);
                }
            }
            // ---- (3) leaves: the nearest of the leaf's triangles ends the search of this mesh, wherever the hit lies.  The pending
            // leaves of the warp are tested COOPERATIVELY: their (ray, triangle) pairs are dealt out over all 32 lanes — a lane
            // fetches the owner's ray by shuffle, tests one triangle, and a segmented min hands the nearest hit (lowest triangle
            // on ties, like the reference's strict '<') back to the owner.  (A loop per owner ran with 6 of 32 lanes.)
            if (__any_sync(0xffffffffu, phase == OCT_LEAF)) {
                const bool owner_lane = phase == OCT_LEAF;
                const int my_cnt = owner_lane ? leaf_cnt : 0;
                if (COUNT) work[1] += (uint32_t)my_cnt;
                int incl = my_cnt;
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const int v = __shfl_up_sync(0xffffffffu, incl, off);
                    if ((int)lane >= off) incl += v;
                }
                const int total = __shfl_sync(0xffffffffu, incl, 31);
                const int excl = incl - my_cnt;   // first pair of this lane's leaf
                float bt = INFINITY;
                uint32_t bid = PC_NONE;
                for (int base = 0; base < total; base += 32) {
                    const int pair = base + (int)lane;
                    int own = 0;   // the last lane whose first pair is <= pair: the owner (lanes without a leaf share the NEXT owner's value)
#pragma unroll
                    for (int step = 16; step; step >>= 1) {
                        const int cand = own + step;
                        const int e = __shfl_sync(0xffffffffu, excl, cand & 31);
                        if (e <= pair) own = cand;
                    }
                    const int k_in = pair - __shfl_sync(0xffffffffu, excl, own);
                    const float3 ro = f3(__shfl_sync(0xffffffffu, o.x, own), __shfl_sync(0xffffffffu, o.y, own), __shfl_sync(0xffffffffu, o.z, own));
                    const float3 rd = f3(__shfl_sync(0xffffffffu, d.x, own), __shfl_sync(0xffffffffu, d.y, own), __shfl_sync(0xffffffffu, d.z, own));
                    const uint32_t rorigin = __shfl_sync(0xffffffffu, origin, own);
                    const int rfirst = __shfl_sync(0xffffffffu, leaf_first, own);
                    float t = INFINITY;
                    uint32_t id = PC_NONE;
                    if (pair < total) {
                        float tt;
                        uint32_t ii;
                        if (oct_tri_test(a.S, rfirst + k_in, ro, rd, rorigin, tt, ii)) { t = tt; id = ii; }
                    }
                    // segmented min towards the first lane of each owner's run (pairs of one owner are neighbours, in triangle order)
#pragma unroll
                    for (int off = 1; off < 32; off <<= 1) {
                        const float t2 = __shfl_down_sync(0xffffffffu, t, off);
                        const uint32_t i2 = __shfl_down_sync(0xffffffffu, id, off);
                        const int o2 = __shfl_down_sync(0xffffffffu, own, off);
                        if ((int)lane + off < 32 && o2 == own && t2 < t) { t = t2; id = i2; }
                    }
                    // the owner reads its run's first lane of this pass (its run may have started in an earlier pass)
                    const int src = max(excl - base, 0);
                    const float ts = __shfl_sync(0xffffffffu, t, src & 31);
                    const uint32_t is = __shfl_sync(0xffffffffu, id, src & 31);
                    if (owner_lane && excl < base + 32 && excl + my_cnt > base && ts < bt) { bt = ts; bid = is; }
                }
                if (owner_lane) {
                    if (bid != PC_NONE) {
                        if (bt < best_t) {   // strict '<' against the best so far (src/scene.rs:280)
                            best_t = bt;
                            best_id = bid;
                        }
                        phase = OCT_NEXT_MESH;
                    } else phase = level < 0 ? OCT_NEXT_MESH : OCT_DESCEND;
                }
            }
            const unsigned act = __ballot_sync(0xffffffffu, phase != OCT_DONE && phase != OCT_IDLE);
            if (act == 0 || (!exhausted && __popc(act) < refill_below)) break;
        }
    }
    if (COUNT) {
        for (int off = 16; off; off >>= 1) {
            work[0] += __shfl_down_sync(0xffffffffu, work[0], off);
            work[1] += __shfl_down_sync(0xffffffffu, work[1], off);
        }
        if (lane == 0) {
            atomicAdd(&C->node_visits, (unsigned long long)work[0]);
            atomicAdd(&C->tri_tests, (unsigned long long)work[1]);
        }
    }
}

// Output slots of k_shade: a warp reserves SHADE_SEG slots of a queue class with ONE atomic and hands them out
// to its lanes over the following trips with warp-local arithmetic; the next segment is reserved while the
// current one still has room for two trips, so the atomic's round trip is never waited for.  (Exact per-trip
// reservations cost one global atomic per warp and trip, whose latency the warp ends up waiting for.)  The slots
// left over when the kernel ends are marked as holes (HIT_HOLE / TLIM_HOLE), which the consumers skip.
// All arguments but `lane` are warp-uniform; lane `cls` keeps the base of the reserved-ahead segment in `nb`.
// DIR = +1: slots grow upward from the returned counter value; -1: downward (back class of the path queue).
template <int DIR>
__device__ __forceinline__ uint32_t seg_alloc(uint32_t& base, uint32_t& used, bool& has_next, uint32_t& nb, unsigned cls,
                                              uint32_t* ctr, unsigned mask, unsigned lane) {
    const uint32_t n = __popc(mask);
    const uint32_t r = used + __popc(mask & ((1u << lane) - 1u));
    const uint32_t step = (uint32_t)(DIR * (int)SHADE_SEG);
    uint32_t slot;
    if (used + n > SHADE_SEG) {   // runs over into the next segment
        if (!has_next && lane == cls) nb = atomic_add_lane(ctr, step);
        uint32_t nbase = __shfl_sync(0xffffffffu, nb, cls);
        if (DIR < 0) nbase -= 1u;   // element 0 of a downward segment sits just below the old tail
        slot = r < SHADE_SEG ? base + (uint32_t)(DIR * (int)r) : nbase + (uint32_t)(DIR * (int)(r - SHADE_SEG));
        base = nbase;
        used = used + n - SHADE_SEG;
        has_next = false;
    } else {
        slot = base + (uint32_t)(DIR * (int)r);
        used += n;
    }
    if (!has_next && used + 64u > SHADE_SEG) {
        if (lane == cls) nb = atomic_add_lane(ctr, step);
        has_next = true;
    }
    return slot;
}
// element k of the segment whose element 0 is `base`
template <int DIR>
__device__ __forceinline__ uint32_t seg_slot(uint32_t base, uint32_t k) { return base + (uint32_t)(DIR * (int)k); }

// ---------------------------------------------------------------- k_shade
// Everything of reflected_radiance except the mesh traversal, as a PERSISTENT kernel of independent warps (no
// CTA barrier after the table staging).  A lane keeps its path IN REGISTERS from vertex to vertex for as long as
// the next nearest hit is already final after the analytic pass (the extension ray cannot reach the mesh box):
// the recursion of src/scene.rs:161-244 becomes a loop, and only rays that need k_traverse go through a queue —
//   * extension ray reaches the mesh box        -> front class of the other path queue, lane takes a new path
//   * NEE candidate reaches the mesh box        -> shadow queue; the path itself is then parked in the back class
//     (at most ONE shadow entry and ONE path entry per input path and iteration: the queue capacities hold)
//   * path ends (roulette, dead surface, miss)  -> lane takes a new path
// New paths come from the current queue: a warp owns one static chunk of SHADE_CHUNK entries and then reserves
// further chunks from a work cursor one chunk ahead; every lane holds one PREFETCHED entry (in shared memory, filled by
// per-thread cp.async copies), so the (streaming) queue loads of a new path are issued a whole trip before they are needed.
// MESH = false: the scene has no triangles — the box tests and the front / shadow queue code vanish at compile time.
// NP > 0: the scene has exactly NP planes + NS spheres (<= 8) and its table rides in the kernel parameters (SmallScene);
// NP = 8, NS = 0: any scene with <= 8 analytic primitives (generic 8-slot form, run-time counts).
// MODE 1 / 2 (FAST) = the reference scenes' case, resolved at compile time: Diffuse / Specular materials only, sphere
// light, no probe items; 1 = live NEE estimator, 2 = the dead "MIS" branch.  MODE 0, the general instantiation, keeps
// every branch at run time (both estimators, Phong, mesh lights, rtb_sample_radiance probes).
constexpr int SHADE_THREADS_NOMESH = 160;   // the mesh-less instantiation needs 96 registers: 4 CTAs of 160 threads = 20 warps per SM
// INLINE = true (the TAIL of a run, launched by the host once few paths are left): a ray that needs the LBVH is traversed right
// here (bvh_traverse, intersect.cuh) instead of being queued for k_traverse, so every remaining path runs to its end inside ONE
// launch — the ~100 iterations in which the last long paths used to die out a few hundred at a time (each four launches that
// hardly fill an SM) collapse into one.  SIMD utilisation of the inline traversal is poor, but the tail holds < 0.1 % of the work.
template <int MODE, int NP = 0, int NS = 0, bool MESH = true, int THREADS = SHADE_THREADS, bool INLINE = false>
__global__ void __launch_bounds__(THREADS, THREADS == SHADE_THREADS ? RTB_SHADE_MINB : 640 / THREADS) k_shade(const __grid_constant__ RenderArgs a, int c) {
    constexpr bool FAST = MODE != 0;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    DevCtrl* C = a.ctrl;
    const DevSceneHeader* hdr = a.S.hdr;
    const uint32_t head = C->ext_head(c), tail = C->ext_tail(c);
    const uint32_t count = head + (a.Pcap - tail);
    if (blockIdx.x * (THREADS / 32) * SHADE_CHUNK >= count) return;   // CTA beyond the static region of a small launch
    const SharedScene sh = stage_scene(a.S, smem_raw, INLINE);   // INLINE: + the traversal stack
    const unsigned lane = threadIdx.x & 31;
    const unsigned below = (1u << lane) - 1u;
    const PathQueue &Q = a.qin, &N = a.qout;
    const int light_obj = hdr->light_obj;
    const bool light_is_mesh = FAST ? false : hdr->light_geom == 2;
    const bool mis = MODE == 1 ? false : (MODE == 2 ? true : a.estimator == 1);     // the reference's dead "MIS" branch
    // RTB_EST_MIS_BALANCE (general instantiation only): next-event estimation and the BRDF sample combined with the balance
    // heuristic — what src/scene.rs:187 ("TODO: Do multiple importance sampling properly") asks for.  Diffuse surfaces under
    // a sphere light; Phong surfaces keep plain NEE (the reference's Phong sampler never leaves the local frame, its pdf
    // for a world direction is undefined).  Never used for parity.
    const bool mis2 = FAST ? false : a.estimator == 2;
    const bool probe_mode = FAST ? false : a.probe_px != nullptr;
    const float3 Le = f3(sh.mats[light_obj].emitted);
    const int n_prims = a.S.n_prims, n_planes = a.S.n_planes;
    const ShadowQueue& SQ = a.sqout;
    uint32_t* const ctr_front = &C->ext_head(1 - c);
    uint32_t* const ctr_back = &C->ext_tail(1 - c);
    uint32_t* const ctr_sh = &C->sh_head(1 - c);
    uint32_t n_ext = 0, n_ext_bvh = 0, n_sh = 0, n_sh_bvh = 0, n_queued = 0;
    uint32_t n_sh_inline = 0;   // INLINE: shadow / probe rays traversed here (counted as BVH shadow rays, never pending)
    auto slot_of = [&](uint32_t i) { return i < head ? i : tail + (i - head); };

    // ---- work fetch (warp-uniform): static first chunk, then chunks from the cursor, reserved one ahead
    const uint32_t gwarp = (blockIdx.x * THREADS + threadIdx.x) >> 5;
    uint32_t wnext = min(gwarp * SHADE_CHUNK, count), wend = min(gwarp * SHADE_CHUNK + SHADE_CHUNK, count);
    bool exhausted = count <= a.shade_warps * SHADE_CHUNK;   // no dynamic chunks in a small launch: no atomics at all
    const bool big_launch = count > a.shade_warps * SHADE_CHUNK * 8u;
    uint32_t nbase = 0;                                      // lane 0: base of the chunk reserved ahead
    if (!exhausted && lane == 0) nbase = atomic_add_lane(&C->cursor_shade, SHADE_CHUNK);

    // ---- lane state: the path being shaded (registers) + one prefetched queue entry (shared memory, filled by per-thread
    // asynchronous copies issued a trip before the entry is needed: it costs no registers while it waits)
    __shared__ __align__(16) float4 spare[5][THREADS];   // o | d | beta | triangle normal | hit (8 bytes used)
    const uint32_t sp_o = (uint32_t)__cvta_generic_to_shared(&spare[0][threadIdx.x]);
    constexpr uint32_t SP_D = THREADS * 16u, SP_B = 2u * SP_D, SP_N = 3u * SP_D, SP_H = 4u * SP_D;
    bool cur_valid = false, cont = false, sp_valid = false, sp_nrm = false;
    float2 h2 = make_float2(0.f, __uint_as_float(PC_NONE));
    float4 o4 = make_float4(0, 0, 0, 0), d4 = o4, b4 = o4, tri_n = o4;   // cont: tri_n carries the stale `o` instead
    float4 ev_keep = o4;   // INLINE: a kept path may sit on a triangle, so the stale `o` / MIS pdf needs its own register
    uint32_t cur_slot = 0, sp_slot = 0;
    // output segments (warp-uniform): front / back class of the other path queue, shadow queue
    uint32_t f_base = 0, f_used = SHADE_SEG, b_base = 0, b_used = SHADE_SEG, s_base = 0, s_used = SHADE_SEG;
    bool f_next = false, b_next = false, s_next = false;
    uint32_t nb = 0;           // lane = class: base of the segment reserved ahead
    // A path that queued a shadow ray (or a dead-MIS probe) stays in registers like any other as long as the shadow queue has
    // room: its NEE candidate is resolved by k_traverse on its own (the entry carries contribution and accumulator index).  Once
    // this warp's shadow segments lie beyond SP entries the old rule applies — such a path is parked — which bounds the queue by
    // 2 SP (+ the segment slack): before, about one path in three written to the path queue was there only because of its shadow ray.
    bool sh_tight = false;

    for (;;) {
        // (a) lanes without a path take their prefetched entry
        if (!cur_valid && sp_valid) {
            cp_async_wait_all();
            h2 = lds_f2(sp_o + SP_H);
            o4 = lds_f4(sp_o);
            d4 = lds_f4(sp_o + SP_D);
            b4 = lds_f4(sp_o + SP_B);
            cur_slot = sp_slot;
            const uint32_t idn = __float_as_uint(h2.y);
            if (idn != PC_NONE && idn != HIT_HOLE && idn >= TRI_BASE)
                tri_n = sp_nrm ? lds_f4(sp_o + SP_N) : __ldg(a.S.tri_nrm + (idn - TRI_BASE));
            cur_valid = idn != HIT_HOLE;
            cont = false;
            sp_valid = false;
        }
        // (b) refill the prefetch slot from the warp's chunk
        {
            const unsigned need = __ballot_sync(0xffffffffu, !sp_valid);
            if (need && wnext < wend) {
                const uint32_t my = wnext + __popc(need & below);
                if (!sp_valid && my < wend) {
                    sp_slot = slot_of(my);
                    cp_async8(sp_o + SP_H, Q.hit + sp_slot);
                    cp_async16(sp_o, Q.o + sp_slot);
                    cp_async16(sp_o + SP_D, Q.d + sp_slot);
                    cp_async16(sp_o + SP_B, Q.beta + sp_slot);
                    cp_async_commit();
                    sp_valid = true;
                    sp_nrm = false;
                }
                wnext = min(wnext + (uint32_t)__popc(need), wend);
            }
            if (wnext >= wend && !exhausted) {   // switch to the chunk reserved ahead, reserve the one after it
                const uint32_t b = __shfl_sync(0xffffffffu, nbase, 0);
                if (b >= count) exhausted = true;
                else {
                    wnext = b;
                    wend = min(b + SHADE_CHUNK, count);
                    if (lane == 0) nbase = atomic_add_lane(&C->cursor_shade, SHADE_CHUNK);
                }
            }
        }
        // (c) done when no lane holds a path or a prefetched entry and the queue is drained
        const unsigned have_work = __ballot_sync(0xffffffffu, cur_valid || sp_valid);
        const bool drained = wnext >= wend && exhausted;
        if (have_work == 0 && drained) break;
        // Tail of a large launch: the queue is drained and only a few lanes still follow a path.  Those paths are
        // parked in the back class after this vertex instead of keeping a mostly idle warp (and the whole launch)
        // alive for the rest of their length; the next iteration packs them densely again.
        const bool park = drained && big_launch && __popc(have_work) < SHADE_PARK_BELOW;

        bool ext_push = false, ext_front = false, sh_push = false, pr_push = false;
        // outputs of this vertex; each is written before it is read under the same flag (no zero-fill: 40 registers)
        float4 eo, ed, eb, ev = make_float4(0.f, 0.f, 0.f, 0.f);
        float2 eh;
        float4 so, sd, sc;
        float4 pd, pc;  // probe entry shares `so`
        eo.w = 0.f;     // flags word: tested (PC_STALE_O) whenever ext_push is set

        if (cur_valid) {
            const uint32_t id = __float_as_uint(h2.y);
            if (id != PC_NONE) {
                const float t = h2.x;
                const float3 o = f3(o4), d = f3(d4);
                const uint32_t origin = __float_as_uint(o4.w);
                const uint32_t acc = __float_as_uint(d4.w);
                float3 beta = f3(b4);
                const uint32_t sdw = __float_as_uint(b4.w);
                const uint32_t sample = sdw >> 12, depth = sdw & 0xfffu;
                const HitGeom hg = hit_geometry(sh, o, d, t, id, tri_n);
                const DevMaterial& mat = sh.mats[hg.obj];
                const float3 ovec = (origin & PC_STALE_O) ? (cont ? f3(INLINE ? ev_keep : tri_n) : f3(Q.ov[cur_slot])) : -d;
                const float3 emitted = f3(mat.emitted);
                const bool emits = emitted.x != 0.f || emitted.y != 0.f || emitted.z != 0.f;
                // emission: received_radiance adds emitted(obj0) (src/scene.rs:155); a specular vertex adds
                // emitted(next) un-attenuated and then scales the reflected part by ks/p (src/scene.rs:176-181)
                if (depth == 1u) {
                    if (emits) accum_add(a.accum, acc, beta * emitted);
                } else if (mis2 && (origin & PC_MIS_PENDING)) {
                    // the BRDF sample of the previous (diffuse) vertex reached the sampled light: its emission counts with the
                    // balance weight pdf_brdf / (pdf_brdf + pdf_light), both per solid angle at the previous vertex
                    if (emits && hg.obj == light_obj) {
                        const float pdf_b = cont ? (INLINE ? ev_keep.w : tri_n.w) : Q.ov[cur_slot].w;
                        const float pdf_l = a.light_pdf * (t * t) / fmaxf(dot(hg.n, -d), 1e-20f);
                        accum_add(a.accum, acc, beta * emitted * (pdf_b / (pdf_b + pdf_l)));
                    }
                } else if (origin & PC_SPEC_PENDING) {
                    if (emits) accum_add(a.accum, acc, beta * emitted);
                    const DevMaterial& pm = sh.mats[object_of(a.S, sh, origin & PC_ID_MASK)];
                    const float inv_pp = (depth - 1u) <= 5u ? 1.0f : (1.0f / 0.9f);   // 1 / survival probability of the specular vertex
                    beta = beta * f3(pm.k) * inv_pp;
                }
                const float p = depth <= 5u ? 1.0f : 0.9f;  // MAX_BOUNCES / SURVIVAL_PROBABILITY (src/scene.rs:109-110,164-168)
                const float inv_p = depth <= 5u ? 1.0f : (1.0f / 0.9f);
                const uint32_t pidx = probe_mode && a.pixel_list ? acc >> 2 : acc;   // probe item, or entry of the pixel list
                const uint32_t rng_pixel = probe_mode ? (uint32_t)(a.probe_py[pidx] * a.width + a.probe_px[pidx]) : acc >> 2;
                const bool dead_surface = mat.brdf == 0 && mat.k.x == 0.f && mat.k.y == 0.f && mat.k.z == 0.f;
                const bool dead_path = beta.x == 0.f && beta.y == 0.f && beta.z == 0.f;
                if (!dead_surface && !dead_path && depth < MAX_DEPTH_FIELD) {
                    const VertexRng vr = rng_vertex(rng_pixel, sample, depth, a.keys);
                    // lobe / light-triangle selectors live in block 1 and are only drawn by Phong surfaces / mesh lights
                    float lobe_u = 0.f, select_u = 0.f;
                    if (!FAST && (mat.brdf == 2 || light_is_mesh)) {
                        const float4 r1 = rng_block(rng_pixel, sample, depth, 1u, a.keys);
                        lobe_u = r1.x;
                        select_u = r1.y;
                    }
                    const float4 r0 = make_float4(vr.light_u1, vr.light_u2, vr.rr, select_u);
                    const float4 rb = make_float4(vr.brdf_u1, vr.brdf_u2, lobe_u, 0.f);
                    float3 next_dir = f3(0.f, 0.f, 0.f), sh_dir = f3(0.f, 0.f, 0.f), sh_contrib = f3(0.f, 0.f, 0.f);
                    float sh_tlim = 0.f;
                    bool want_sh = false;
                    if (mat.brdf == 1) {  // specular branch, src/scene.rs:170-185
                        if (r0.z < p) {
                            next_dir = flip_across(ovec, hg.n);
                            ext_push = true;
                            eo = make_float4(hg.pos.x, hg.pos.y, hg.pos.z, __uint_as_float(hg.pcode | PC_SPEC_PENDING | PC_STALE_O));
                            eb = make_float4(beta.x, beta.y, beta.z, __uint_as_float((sample << 12) | (depth + 1u)));
                            ev = make_float4(ovec.x, ovec.y, ovec.z, 0.f);  // the recursion is handed `o`, not -i (src/scene.rs:178)
                        }
                    } else {
                        // ---- direct light
                        float3 y, ny;
                        float pdf_a;
                        if (FAST) light_sample_sphere(a.light_sphere, a.light_pdf, r0, y, ny, pdf_a);
                        else light_sample<FAST>(a.S, sh.prims, hdr, r0, y, ny, pdf_a);
                        float3 dv = y - hg.pos;
                        float r2 = dot(dv, dv);
                        float inv_dist = rsqrtf(r2);
                        float dist = r2 * inv_dist;
                        float3 inc = dv * inv_dist;
                        float3 f = brdf_eval<FAST>(mat, hg.n, ovec, inc);
                        float3 contrib;
                        if (!mis) {  // live NEE, src/scene.rs:217-229 (no cosine is clamped)
                            float g = __fdividef(dot(hg.n, inc) * dot(ny, -inc), r2 * pdf_a);
                            contrib = beta * Le * f * g;
                            if (mis2 && mat.brdf == 0) {   // balance weight of the light sample: pdf_light / (pdf_light + pdf_brdf(inc))
                                const float pdf_l = pdf_a * r2 / fmaxf(fabsf(dot(ny, -inc)), 1e-20f);
                                const float pdf_b = fmaxf(dot(hg.n, inc), 0.f) * INV_PI_F;
                                contrib = contrib * (pdf_l / (pdf_l + pdf_b));
                            }
                        } else {                 // dead branch, src/scene.rs:191-201
                            float pdf_light = pdf_a * (r2 / dot(ny, -inc));
                            float3 itmp;
                            float pdf_fresh;
                            brdf_sample<FAST>(mat, hg.n, inc, rng_block(rng_pixel, sample, depth, 2u, a.keys), itmp, pdf_fresh);
                            contrib = beta * Le * f * (dot(hg.n, inc) / (pdf_light + pdf_fresh));
                        }
                        if (contrib.x != 0.f || contrib.y != 0.f || contrib.z != 0.f) {
                            want_sh = true;     // mutually_visible is resolved below, together with the extension ray
                            sh_dir = inc;
                            sh_tlim = dist - SHADOW_MARGIN;
                            sh_contrib = contrib;
                            ++n_sh;
                        }
                        if (mis) {  // src/scene.rs:203-214: own BRDF sample; counts only if it reaches the light
                            float3 i2;
                            float pdf2;
                            brdf_sample<FAST>(mat, hg.n, ovec, rng_block(rng_pixel, sample, depth, 4u, a.keys), i2, pdf2);
                            if (i2.x != 0.f || i2.y != 0.f || i2.z != 0.f) {
                                float3 y2, ny2;
                                float pdf_a2;
                                if (FAST) light_sample_sphere(a.light_sphere, a.light_pdf, rng_block(rng_pixel, sample, depth, 3u, a.keys), y2, ny2, pdf_a2);
                                else light_sample<FAST>(a.S, sh.prims, hdr, rng_block(rng_pixel, sample, depth, 3u, a.keys), y2, ny2, pdf_a2);
                                float3 dv2 = y2 - hg.pos;
                                float pdf_light2 = pdf_a2 * (dot(dv2, dv2) / dot(ny2, -i2));
                                float3 c2 = beta * Le * brdf_eval<FAST>(mat, hg.n, ovec, i2) * (dot(hg.n, i2) / (pdf2 + pdf_light2));
                                if (c2.x != 0.f || c2.y != 0.f || c2.z != 0.f) {
                                    // trace_ray(x, i2) and test hit.id == light_source
                                    ++n_sh;
                                    float ta;
                                    uint32_t ida;
                                    if (NP > 0 && NP < 8) analytic_closest_small<NP, NS>(a.ss, origin_group_of(sh, hg.pcode), hg.pos, i2, hg.pcode, ta, ida);
                                    else analytic_closest(sh, n_planes, n_prims, hg.pos, i2, hg.pcode, ta, ida);
                                    const bool needs_bvh = MESH ? ray_hits_bvh_box(a.S, hg.pos, i2, ta) : false;
                                    if (!light_is_mesh) {
                                        // the light is analytic: it must be the nearest analytic hit and no triangle may lie in front of it
                                        if (ida != PC_NONE && sh.prims[ida].obj == light_obj) {
                                            if (needs_bvh && INLINE) {
                                                ++n_sh_inline;
                                                uint32_t idt = PC_NONE;
                                                float tt = ta;
                                                if (!bvh_traverse<true, false>(a.S, sh, hg.pos, i2, hg.pcode, tt, idt, ta + SHADOW_MARGIN, nullptr)) accum_add(a.accum, acc, c2);
                                            } else if (needs_bvh) {
                                                pr_push = true;
                                                pd = make_float4(i2.x, i2.y, i2.z, ta);
                                                pc = make_float4(c2.x, c2.y, c2.z, __uint_as_float(acc));
                                            } else {
                                                accum_add(a.accum, acc, c2);
                                            }
                                        }
                                    } else if (needs_bvh && INLINE) {   // mesh light, traversed here: see below
                                        ++n_sh_inline;
                                        uint32_t idt = PC_NONE;
                                        float tt = ta;
                                        bvh_traverse<false, false>(a.S, sh, hg.pos, i2, hg.pcode, tt, idt, 0.f, nullptr);
                                        if (idt != PC_NONE && __float_as_int(__ldg(a.S.tris + (size_t)(idt - TRI_BASE) * TRI_STRIDE + 2).w) == light_obj) accum_add(a.accum, acc, c2);
                                    } else if (needs_bvh) {  // mesh light: nearest triangle below the analytic hit must belong to it
                                        pr_push = true;
                                        pd = make_float4(i2.x, i2.y, i2.z, ta);
                                        pc = make_float4(c2.x, c2.y, c2.z, __uint_as_float(acc | SHADOW_PROBE));
                                    }
                                    if (pr_push) {
                                        ++n_sh_bvh;
                                        so = make_float4(hg.pos.x, hg.pos.y, hg.pos.z, __uint_as_float(hg.pcode));
                                    }
                                }
                            }
                        }
                        // ---- russian roulette + continuation, src/scene.rs:231-240
                        if (r0.z < p) {
                            float pdf1;
                            brdf_sample<FAST>(mat, hg.n, ovec, rb, next_dir, pdf1);
                            if (next_dir.x != 0.f || next_dir.y != 0.f || next_dir.z != 0.f) {
                                float3 nb;
                                if (FAST || mat.brdf == 0) nb = beta * f3(mat.k) * inv_p;  // f (n.i) / pdf == kd exactly
                                else nb = beta * brdf_eval(mat, hg.n, ovec, next_dir) * (dot(hg.n, next_dir) / (pdf1 * p));
                                ext_push = true;
                                eo = make_float4(hg.pos.x, hg.pos.y, hg.pos.z, __uint_as_float(hg.pcode));
                                eb = make_float4(nb.x, nb.y, nb.z, __uint_as_float((sample << 12) | (depth + 1u)));
                                if (mis2 && mat.brdf == 0) {   // the sample's pdf travels with the ray (see PC_MIS_PENDING)
                                    eo.w = __uint_as_float(hg.pcode | PC_MIS_PENDING);
                                    ev = make_float4(0.f, 0.f, 0.f, pdf1);
                                }
                            }
                        }
                    }
                    if (ext_push || want_sh) {
                        // Analytic half of BOTH trace_ray calls this vertex makes (extension: nearest hit; shadow:
                        // mutually_visible, src/scene.rs:258-270), here where every lane does it together.  Rays that
                        // can still reach the mesh box afterwards are queued for k_traverse.
                        float ta;
                        uint32_t ida;
                        bool occ;
                        if (NP == 8) analytic_pair_small8(a.ss, n_planes, n_prims, origin_group_of(sh, hg.pcode), hg.pos, hg.pcode, next_dir, ta, ida, sh_dir, sh_tlim, occ);
                        else if (NP > 0) analytic_pair_small<NP, NS>(a.ss, origin_group_of(sh, hg.pcode), hg.pos, hg.pcode, next_dir, ta, ida, sh_dir, sh_tlim, occ);
                        else analytic_pair(sh, n_planes, n_prims, hg.pos, hg.pcode, next_dir, ta, ida, sh_dir, sh_tlim, occ);
                        bool ext_box, sh_box;   // can the two rays still reach the mesh box?  (both at once: shared terms, packed products)
                        if (MESH) ray_pair_hits_bvh_box(a.S, hg.pos, next_dir, ta, sh_dir, sh_tlim, ext_box, sh_box);
                        else ext_box = sh_box = false;   // no triangles in the scene: no ray ever leaves this kernel for k_traverse
                        if (want_sh && !occ) {
                            if (sh_box && INLINE) {   // mutually_visible's mesh half, right here
                                ++n_sh_inline;
                                uint32_t idt = PC_NONE;
                                float tt = sh_tlim;
                                if (!bvh_traverse<true, false>(a.S, sh, hg.pos, sh_dir, hg.pcode, tt, idt, sh_tlim + SHADOW_MARGIN, nullptr)) accum_add(a.accum, acc, sh_contrib);
                            } else if (sh_box) {
                                sh_push = true;
                                ++n_sh_bvh;
                                so = make_float4(hg.pos.x, hg.pos.y, hg.pos.z, __uint_as_float(hg.pcode));
                                sd = make_float4(sh_dir.x, sh_dir.y, sh_dir.z, sh_tlim);
                                sc = make_float4(sh_contrib.x, sh_contrib.y, sh_contrib.z, __uint_as_float(acc));
                            } else {
                                accum_add(a.accum, acc, sh_contrib);
                            }
                        }
                        if (ext_push) {
                            ext_front = ext_box;
                            n_ext_bvh += ext_front ? 1u : 0u;
                            if (INLINE && ext_front) {   // Mesh::intersect for the extension ray, right here: the hit is final afterwards
                                bvh_traverse<false, false>(a.S, sh, hg.pos, next_dir, hg.pcode, ta, ida, 0.f, nullptr);
                                ext_front = false;
                            }
                            ed = make_float4(next_dir.x, next_dir.y, next_dir.z, __uint_as_float(acc));
                            eh = make_float2(ta, __uint_as_float(ida));
                            ++n_ext;
                        }
                    }
                }
            }
        }
        // ---- where does the path go?  In registers if its next hit is final and it queued no shadow ray.
        bool keep = ext_push && !ext_front && !park && (!(sh_push || pr_push) || !sh_tight);
        if (ext_push && !ext_front && __float_as_uint(eh.y) == PC_NONE) {   // left the scene: nothing to shade
            keep = false;
            ext_push = false;
        }
        if (keep) ext_push = false;
        // ---- queue pushes: slots from the warp's segments (see seg_alloc), written straight away
        const unsigned mf = __ballot_sync(0xffffffffu, ext_push && ext_front);
        const unsigned mb = __ballot_sync(0xffffffffu, ext_push && !ext_front);
        const unsigned ms = __ballot_sync(0xffffffffu, sh_push);
        const unsigned mp = __ballot_sync(0xffffffffu, pr_push);
        if (mf | mb) {
            uint32_t slot = 0;
            if (mf) { const uint32_t v = seg_alloc<1>(f_base, f_used, f_next, nb, 0u, ctr_front, mf, lane); if (ext_front) slot = v; }
            if (mb) { const uint32_t v = seg_alloc<-1>(b_base, b_used, b_next, nb, 1u, ctr_back, mb, lane); if (!ext_front) slot = v; }
            if (ext_push && slot >= a.Pcap) { atomicAdd(&C->overflow, 1u); ext_push = false; }
            if (ext_push) {
                N.o[slot] = eo;
                N.d[slot] = ed;
                N.beta[slot] = eb;
                N.hit[slot] = eh;
                if (__float_as_uint(eo.w) & (PC_STALE_O | PC_MIS_PENDING)) N.ov[slot] = ev;
                ++n_queued;
            }
        }
        if (ms) {
            const uint32_t slot = seg_alloc<1>(s_base, s_used, s_next, nb, 2u, ctr_sh, ms, lane);
            if (sh_push && slot >= a.SPcap) { atomicAdd(&C->overflow, 1u); sh_push = false; }
            if (sh_push) { SQ.o[slot] = so; SQ.d[slot] = sd; SQ.c[slot] = sc; }
        }
        if (mp) {
            const uint32_t slot = seg_alloc<1>(s_base, s_used, s_next, nb, 2u, ctr_sh, mp, lane);
            if (pr_push && slot >= a.SPcap) { atomicAdd(&C->overflow, 1u); pr_push = false; }
            if (pr_push) { SQ.o[slot] = so; SQ.d[slot] = pd; SQ.c[slot] = pc; }
        }
        if (ms | mp) sh_tight = s_base + SHADE_SEG > a.SP;   // warp-uniform: where this warp's current shadow segment ends
        // ---- next vertex of the same path, straight from registers
        cur_valid = keep;
        if (keep) {
            o4 = eo; d4 = ed; b4 = eb; h2 = eh;
            if (INLINE) {    // the next hit may be a triangle (traversed above): its normal, and the stale `o` in its own register
                ev_keep = ev;
                const uint32_t idk = __float_as_uint(eh.y);
                if (idk != PC_NONE && idk >= TRI_BASE) tri_n = __ldg(a.S.tri_nrm + (idk - TRI_BASE));
            } else {
                tri_n = ev;  // stale `o` of a specular vertex (PC_STALE_O in eo.w); analytic hits need no triangle normal
            }
            cont = true;
        }
        // ---- the prefetched entry's hit id has arrived by now -> start the dependent triangle-normal fetch
        if (sp_valid && !sp_nrm) {
            cp_async_wait_all();
            const uint32_t idn = __float_as_uint(lds_f2(sp_o + SP_H).y);
            if (idn == HIT_HOLE) sp_valid = false;   // unfilled slot of the producer: ask for another entry next trip
            else if (idn != PC_NONE && idn >= TRI_BASE) {
                cp_async16(sp_o + SP_N, a.S.tri_nrm + (idn - TRI_BASE));
                cp_async_commit();
            }
            sp_nrm = true;
        }
    }
    // epilogue: mark the slots this warp reserved but did not fill
    {
        const float2 hole = make_float2(0.f, __uint_as_float(HIT_HOLE));
        const float4 hole4 = make_float4(0.f, 0.f, 0.f, __uint_as_float(TLIM_HOLE));
        auto mark_path = [&](uint32_t slot) { if (slot < a.Pcap) N.hit[slot] = hole; else atomicAdd(&C->overflow, 1u); };
        auto mark_sh = [&](uint32_t slot) { if (slot < a.SPcap) SQ.d[slot] = hole4; else atomicAdd(&C->overflow, 1u); };
        for (uint32_t k = f_used + lane; k < SHADE_SEG; k += 32) mark_path(seg_slot<1>(f_base, k));
        for (uint32_t k = b_used + lane; k < SHADE_SEG; k += 32) mark_path(seg_slot<-1>(b_base, k));
        for (uint32_t k = s_used + lane; k < SHADE_SEG; k += 32) mark_sh(seg_slot<1>(s_base, k));
        const uint32_t nf = __shfl_sync(0xffffffffu, nb, 0), nbk = __shfl_sync(0xffffffffu, nb, 1) - 1u, ns = __shfl_sync(0xffffffffu, nb, 2);
        if (f_next) for (uint32_t k = lane; k < SHADE_SEG; k += 32) mark_path(seg_slot<1>(nf, k));
        if (b_next) for (uint32_t k = lane; k < SHADE_SEG; k += 32) mark_path(seg_slot<-1>(nbk, k));
        if (s_next) for (uint32_t k = lane; k < SHADE_SEG; k += 32) mark_sh(seg_slot<1>(ns, k));
    }
    // counters
    for (int off = 16; off; off >>= 1) {
        n_ext += __shfl_down_sync(0xffffffffu, n_ext, off);
        n_ext_bvh += __shfl_down_sync(0xffffffffu, n_ext_bvh, off);
        n_sh += __shfl_down_sync(0xffffffffu, n_sh, off);
        n_sh_bvh += __shfl_down_sync(0xffffffffu, n_sh_bvh, off);
        if (INLINE) n_sh_inline += __shfl_down_sync(0xffffffffu, n_sh_inline, off);
        n_queued += __shfl_down_sync(0xffffffffu, n_queued, off);
    }
    if (lane == 0) {
        if (n_queued) { atomicAdd(&C->live[1 - c], n_queued); atomicAdd(&C->paths_queued, (unsigned long long)n_queued); }
        if (n_sh_bvh) atomicAdd(&C->sh_live[1 - c], n_sh_bvh);
        if (n_ext) atomicAdd(&C->rays_extension, (unsigned long long)n_ext);
        if (n_ext_bvh) atomicAdd(&C->rays_bvh, (unsigned long long)n_ext_bvh);
        if (n_sh) atomicAdd(&C->rays_shadow, (unsigned long long)n_sh);
        if (n_sh_bvh + n_sh_inline) atomicAdd(&C->shadow_bvh, (unsigned long long)(n_sh_bvh + n_sh_inline));
    }
}

// ---------------------------------------------------------------- k_resolve
// sample_pixel's tail (src/server.rs:360-363) + gamma_correct (:366-368) + `as u8` (:187-189):
// per sub-pixel mean -> clamp -> *0.25 -> sum -> clamp -> ^(1/2.2) * 255 + 0.5 -> truncate.
__device__ __forceinline__ float clamp01_keep_nan(float x) { return x < 0.f ? 0.f : (x > 1.f ? 1.f : x); }
__device__ __forceinline__ unsigned char to_u8(float v) {
    if (!(v == v)) return 0;  // Rust `as u8`: NaN -> 0, saturating, truncating
    if (v <= 0.f) return 0;
    if (v >= 255.f) return 255;
    return (unsigned char)v;
}

// scanline 0: out_rgb8 in tile order (lp*3); 1: scan-line frame (y*width + x)*3
__global__ void k_resolve(RenderArgs a, unsigned char* __restrict__ out_rgb8, float4* __restrict__ out_sub, int scanline) {
    int lp = blockIdx.x * blockDim.x + threadIdx.x;
    if (lp >= a.n_local_tiles * 1024) return;
    int x, y;
    bool in = local_to_xy(lp + a.tile_base * 1024, a.rank, a.world, a.tiles_x, a.width, a.height, x, y);
    float3 px = f3(0.f, 0.f, 0.f);
    if (in) {
        uint32_t p = (uint32_t)(y * a.width + x);
        const uint32_t ks_done = a.tile_ks ? a.tile_ks[(lp >> 10) + a.tile_base] : a.ks_done;
        for (int s = 0; s < 4; ++s) {
            // sub-pixel s has received the samples ks < ks_done with ks % 4 == s
            uint32_t cnt = ks_done > (uint32_t)s ? (ks_done - (uint32_t)s + 3u) / 4u : 0u;
            float inv = cnt ? 1.0f / (float)cnt : 0.0f;
            float4 v = a.accum[p * 4u + s];
            if (out_sub) out_sub[(size_t)lp * 4 + s] = make_float4(v.x * inv, v.y * inv, v.z * inv, 0.f);
            px.x += clamp01_keep_nan(v.x * inv) * 0.25f;
            px.y += clamp01_keep_nan(v.y * inv) * 0.25f;
            px.z += clamp01_keep_nan(v.z * inv) * 0.25f;
        }
    } else if (out_sub) {
        for (int s = 0; s < 4; ++s) out_sub[(size_t)lp * 4 + s] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
    unsigned char r = to_u8(powf(clamp01_keep_nan(px.x), 1.0f / 2.2f) * 255.0f + 0.5f);
    unsigned char g = to_u8(powf(clamp01_keep_nan(px.y), 1.0f / 2.2f) * 255.0f + 0.5f);
    unsigned char b = to_u8(powf(clamp01_keep_nan(px.z), 1.0f / 2.2f) * 255.0f + 0.5f);
    if (scanline) {
        if (!in) return;
        size_t o = ((size_t)y * a.width + x) * 3;
        out_rgb8[o] = r; out_rgb8[o + 1] = g; out_rgb8[o + 2] = b;
    } else {
        size_t o = (size_t)lp * 3;
        out_rgb8[o] = in ? r : 0; out_rgb8[o + 1] = in ? g : 0; out_rgb8[o + 2] = in ? b : 0;
    }
}

// sample_pixel's return value for a LIST of pixels (rtb_sample_pixels): accumulators [i*4 + sub] -> Vec3 in 0..255.5, i.e.
// gamma_correct applied, before RenderJob::run's `as u8` (src/server.rs:360-368)
__global__ void k_resolve_list(const float4* __restrict__ accum, int n, int num_samples, float* __restrict__ out3) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const float inv = num_samples > 0 ? 1.0f / (float)num_samples : 0.0f;
    float3 px = f3(0.f, 0.f, 0.f);
    for (int s = 0; s < 4; ++s) {
        const float4 v = accum[(size_t)i * 4 + s];
        px.x += clamp01_keep_nan(v.x * inv) * 0.25f;
        px.y += clamp01_keep_nan(v.y * inv) * 0.25f;
        px.z += clamp01_keep_nan(v.z * inv) * 0.25f;
    }
    out3[3 * i] = powf(clamp01_keep_nan(px.x), 1.0f / 2.2f) * 255.0f + 0.5f;
    out3[3 * i + 1] = powf(clamp01_keep_nan(px.y), 1.0f / 2.2f) * 255.0f + 0.5f;
    out3[3 * i + 2] = powf(clamp01_keep_nan(px.z), 1.0f / 2.2f) * 255.0f + 0.5f;
}

// ---------------------------------------------------------------- adaptive sampling (world = 1)
// A pass renders the tiles of `list` (ascending tile order); k_adapt then updates every pixel's statistic (adapt_pixel),
// decides per tile whether it goes on, and k_compact_tiles squeezes the tiles that stopped out of the list.
struct AdaptArgs {
    float4* accum;       // [pixel*4 + sub]: .w holds lum709 of the sums after the previous pass
    float2* mom;         // [pixel]: (mean, M2) of the batch values
    int32_t* list;       // the pass's tiles; k_adapt marks a tile that stops with -1
    uint32_t* tile_ks;   // [tile]: samples per pixel so far (= ks_done of k_resolve)
    float* tile_err;     // [tile]: max over the tile's pixels of adapt_pixel's error after its latest pass
    int width, height, tiles_x;
    int pass_spp, spp, min_spp;
    float target;        // 8-bit output levels; 0 = never stop before the budget
};

constexpr int ADAPT_THREADS = 256;
constexpr int COMPACT_THREADS = 1024;

__global__ void k_adapt_init(AdaptArgs a, int n_tiles) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tiles) return;
    a.list[t] = t;
    a.tile_ks[t] = 0u;
    a.tile_err[t] = 0.0f;
}

// one CTA per tile of the pass's list
__global__ void __launch_bounds__(ADAPT_THREADS) k_adapt(AdaptArgs a) {
    __shared__ float warp_max[ADAPT_THREADS / 32];
    const int t = a.list[blockIdx.x];
    const uint32_t ks = a.tile_ks[t] + (uint32_t)a.pass_spp;
    const int B = (int)(ks / (uint32_t)a.pass_spp);
    const float inv_n = 4.0f / (float)a.pass_spp;
    float err = 0.0f;
    for (int slot = threadIdx.x; slot < 1024; slot += ADAPT_THREADS) {
        int x, y;
        if (!local_to_xy(t * 1024 + slot, 0, 1, a.tiles_x, a.width, a.height, x, y)) continue;
        const uint32_t p = (uint32_t)(y * a.width + x);
        float4 sub[4];
        for (int s = 0; s < 4; ++s) sub[s] = a.accum[p * 4u + s];
        float2 mom = a.mom[p];
        err = fmaxf(err, adapt_pixel(sub, inv_n, mom, B));
        for (int s = 0; s < 4; ++s) a.accum[p * 4u + s].w = sub[s].w;
        a.mom[p] = mom;
    }
    for (int off = 16; off; off >>= 1) err = fmaxf(err, __shfl_xor_sync(0xffffffffu, err, off));
    if ((threadIdx.x & 31) == 0) warp_max[threadIdx.x >> 5] = err;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < ADAPT_THREADS / 32; ++w) err = fmaxf(err, warp_max[w]);
        a.tile_ks[t] = ks;
        a.tile_err[t] = err;
        const bool go_on = ks < (uint32_t)a.spp && (ks < (uint32_t)a.min_spp || a.target <= 0.0f || err > a.target);
        if (!go_on) a.list[blockIdx.x] = -1;
    }
}

// one CTA: drops the -1 entries of list[0, n) in place, order kept (an entry only ever moves towards the front, and a chunk
// is read completely before any of it is written); the new count goes to mapped host memory
__global__ void __launch_bounds__(COMPACT_THREADS) k_compact_tiles(int32_t* list, int n, volatile int* host_count) {
    __shared__ int warp_sum[COMPACT_THREADS / 32];
    __shared__ int base;
    const unsigned lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    if (threadIdx.x == 0) base = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n; c0 += COMPACT_THREADS) {
        const int i = c0 + (int)threadIdx.x;
        const int32_t v = i < n ? list[i] : -1;
        const unsigned keep = __ballot_sync(0xffffffffu, v >= 0);
        if (lane == 0) warp_sum[w] = __popc(keep);
        __syncthreads();
        int before = base, total = 0;
        for (int k = 0; k < COMPACT_THREADS / 32; ++k) {
            before += k < (int)w ? warp_sum[k] : 0;
            total += warp_sum[k];
        }
        if (v >= 0) list[before + __popc(keep & ((1u << lane) - 1u))] = v;
        __syncthreads();
        if (threadIdx.x == 0) base += total;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        *host_count = base;
        __threadfence_system();
    }
}

// scatter `world` tile-ordered shards into a scan-line frame
__global__ void k_untile(const unsigned char* __restrict__ shards, long long shard_stride, int world, int tiles_x, int tiles_y,
                         int width, int height, unsigned char* __restrict__ frame) {
    long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    long long total = (long long)tiles_x * tiles_y * 1024;
    if (g >= total) return;
    int t = (int)(g >> 10), slot = (int)(g & 1023);
    int rank = t % world, lt = t / world;
    int x, y;
    if (!local_to_xy(lt * 1024 + slot, rank, world, tiles_x, width, height, x, y)) return;
    const unsigned char* s = shards + (size_t)rank * shard_stride + ((size_t)lt * 1024 + slot) * 3;
    size_t o = ((size_t)y * width + x) * 3;
    frame[o] = s[0]; frame[o + 1] = s[1]; frame[o + 2] = s[2];
}

// ---------------------------------------------------------------- parity hook: explicit rays
template <bool COUNT>
__global__ void __launch_bounds__(WF_THREADS) k_trace_rays(DevScene S, long long n, const float* __restrict__ org, const float* __restrict__ dir,
                                                           const Camera cam, int width, int height, int sx, int sy, float dx, float dy,
                                                           int32_t* __restrict__ obj, int32_t* __restrict__ tri, float* __restrict__ tout,
                                                           unsigned long long* __restrict__ work_out, int accel = 0) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SharedScene sh = stage_scene(S, smem_raw);
    uint32_t work[2] = {0, 0};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        float3 o, d;
        if (org) {
            o = f3(org[3 * i], org[3 * i + 1], org[3 * i + 2]);
            d = f3(dir[3 * i], dir[3 * i + 1], dir[3 * i + 2]);
        } else {  // camera rays, row 0 = top of the screen
            int y = (int)(i / width), x = (int)(i - (long long)y * width);
            o = cam.pos;
            d = camera_dir(cam, x, height - y - 1, sx, sy, dx, dy, (float)width, (float)height);
        }
        float t;
        uint32_t id;
        analytic_closest(sh, S.n_planes, S.n_prims, o, d, PC_NONE, t, id);
        if (accel == 1) {   // RTB_ACCEL_OCTREE_REFERENCE
            oct_trace_meshes(S, o, d, PC_NONE, t, id, COUNT ? work : nullptr);
        } else if (ray_hits_bvh_box(S, o, d, t)) {
            if (S.wide) bvh_traverse<false, COUNT, true>(S, sh, o, d, PC_NONE, t, id, 0.0f, work);
            else bvh_traverse<false, COUNT, false>(S, sh, o, d, PC_NONE, t, id, 0.0f, work);
        }
        if (id == PC_NONE) {
            obj[i] = -1; tri[i] = -1; tout[i] = INFINITY;
        } else if (id < TRI_BASE) {
            obj[i] = sh.prims[id].obj; tri[i] = -1; tout[i] = t;
        } else {
            const float4* tp = S.tris + (size_t)(id - TRI_BASE) * TRI_STRIDE;
            int ob = __float_as_int(__ldg(tp + 2).w);
            obj[i] = ob;
            tri[i] = __float_as_int(__ldg(tp + 1).w) - sh.mats[ob].first_tri;
            tout[i] = t;
        }
    }
    if (COUNT && work_out) {
        atomicAdd(&work_out[0], (unsigned long long)work[0]);
        atomicAdd(&work_out[1], (unsigned long long)work[1]);
    }
}

// FP32 peak probe: 8 independent FMA chains per thread
__global__ void k_fma_peak(float* out, int iters) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
    const float m = 0.999f, c = 1e-3f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
            a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}

}  // namespace rtb
