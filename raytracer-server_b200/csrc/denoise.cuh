// denoise.cuh — the opt-in denoiser: guides (k_gbuffer) and the edge-aware à-trous filter (k_denoise_prep, k_atrous,
// k_denoise_out).  The filter rule itself lives in denoise_rule.cuh; DESIGN §3d has the design and the measurements.
//
// Whole frames only (world = 1): every buffer is in scan-line order, row 0 = top.
#pragma once

#include "denoise_rule.cuh"
#include "wavefront.cuh"

namespace rtb {

constexpr int GBUFFER_MAX_BOUNCES = 8;   // specular bounces a guide ray follows
constexpr int DENOISE_THREADS = 256;

// ---------------------------------------------------------------- guides
// For each pixel the four sub-pixel centre rays (those of rtb_trace_primary(sx, sy, 0, 0)), each followed through up to
// GBUFFER_MAX_BOUNCES specular vertices in the direction k_shade takes there (the stale-`o` quirk included: every vertex
// of a chain reflects the camera ray's -d).  Per ray: the first non-specular hit's object, facing normal, path length and
// albedo (times ks of every mirror on the way); an emitter, a miss or an unfinished chain has albedo 1.  Per pixel:
// A dielectric counts as a specular vertex: the ray follows the refracted direction (the reflected one under total internal
// reflection) and the albedo takes the tint on transmission.  A rough metal (brdf 4) is a non-specular first hit of albedo F0.
// ga = (mean albedo, mean depth over the rays that hit), gn = (renormalised sum of the normals, the object most rays hit,
// ties to the lowest sub-pixel; -1 = miss).
__global__ void __launch_bounds__(WF_THREADS) k_gbuffer(DevScene S, const Camera cam, int width, int height, int accel,
                                                        float4* __restrict__ ga, float4* __restrict__ gn) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const SharedScene sh = stage_scene(S, smem_raw);
    const long long n = (long long)width * height;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const int y = (int)(i / width), x = (int)(i - (long long)y * width);
        float3 alb = f3(0.f, 0.f, 0.f), nrm = f3(0.f, 0.f, 0.f);
        float depth = 0.f;
        int hits = 0;
        int objs[4];
        for (int s = 0; s < 4; ++s) {
            float3 o = cam.pos, d = camera_dir(cam, x, height - y - 1, s & 1, s >> 1, 0.f, 0.f, (float)width, (float)height);
            uint32_t origin = PC_NONE;
            float3 thr = f3(1.f, 1.f, 1.f), ovec = -d;
            float path = 0.f;
            int obj = -1;
            float3 a = f3(1.f, 1.f, 1.f);
            for (int b = 0; b <= GBUFFER_MAX_BOUNCES; ++b) {
                float t;
                uint32_t id;
                analytic_closest(sh, S.n_planes, S.n_prims, o, d, origin, t, id);
                if (accel == 1) oct_trace_meshes(S, o, d, origin, t, id, nullptr);   // RTB_ACCEL_OCTREE_REFERENCE
                else if (ray_hits_bvh_box(S, o, d, t)) bvh_traverse<false, false>(S, sh, o, d, origin, t, id, 0.0f, nullptr);
                if (id == PC_NONE) { obj = -1; break; }
                path += t;
                const float4 tri_n = id >= TRI_BASE ? __ldg(S.tri_nrm + (id - TRI_BASE)) : make_float4(0.f, 0.f, 0.f, 0.f);
                const HitGeom hg = hit_geometry(sh, o, d, t, id, tri_n);
                const DevMaterial& m = sh.mats[hg.obj];
                obj = hg.obj;
                if (m.brdf == 1 && b < GBUFFER_MAX_BOUNCES) {   // specular: src/scene.rs:170-185 hands the recursion `o`, not -i
                    thr = thr * f3(m.k);
                    d = flip_across(ovec, hg.n);
                    o = hg.pos;
                    origin = hg.pcode;
                    continue;
                }
                if (m.brdf == 3 && b < GBUFFER_MAX_BOUNCES) {   // dielectric: refract, or reflect under total internal reflection
                    const bool flipped = (hg.pcode & PC_FLIPPED) != 0u;
                    float cos_t;
                    const float F = dielectric_fresnel(-dot(d, hg.n), dielectric_entering(flipped, m.k.y) ? 1.0f / m.k.x : m.k.x, cos_t);
                    bool refracted;
                    d = dielectric_scatter(d, hg.n, flipped, m.k.y, m.k.x, F < 1.0f ? 1.0f : 0.0f, refracted);
                    ovec = -d;   // the stale-`o` quirk restarts from the true direction, as in k_shade
                    o = hg.pos;
                    origin = hg.pcode;
                    if (refracted) {   // k_shade's rule: leave through the other side
                        origin ^= PC_FLIPPED;
                        if (m.geom != 0) o = hg.pos - (2.0f * SURF_OFFSET) * hg.n;
                        thr = thr * f3(m.color_d);
                    }
                    continue;
                }
                const bool emits = m.emitted.x != 0.f || m.emitted.y != 0.f || m.emitted.z != 0.f;
                if (m.brdf == 4 && !emits) a = thr * f3(m.color_s);   // rough metal: F0
                else if (m.brdf != 1 && m.brdf != 3 && !emits)
                    a = thr * (m.brdf == 0 ? f3(m.k) : f3(m.color_d) * m.k.x + f3(m.color_s) * m.k.y);
                nrm = nrm + hg.n;
                depth += path;
                ++hits;
                break;
            }
            alb = alb + a;
            objs[s] = obj;
        }
        int best = objs[0], best_n = 0;
        for (int s = 0; s < 4; ++s) {
            int c = 0;
            for (int k = 0; k < 4; ++k) c += objs[k] == objs[s];
            if (c > best_n) { best = objs[s]; best_n = c; }
        }
        const float len2 = dot(nrm, nrm);
        if (len2 > 0.f) nrm = nrm * rsqrtf(len2);
        ga[i] = make_float4(alb.x * 0.25f, alb.y * 0.25f, alb.z * 0.25f, hits ? depth / (float)hits : 0.f);
        gn[i] = make_float4(nrm.x, nrm.y, nrm.z, __int_as_float(best));
    }
}

// ---------------------------------------------------------------- filter
struct DenoiseArgs {
    const float4* accum;      // [pixel*4 + sub] rgb sums; nullptr: rtb_denoise_image, buf[1] holds (colour rgb, variance)
    uint32_t ks_done;         // as RenderArgs::ks_done / tile_ks: the samples each sub-pixel has received
    const uint32_t* tile_ks;
    int tiles_x;
    int width, height;
    const float4* ga;
    const float4* gn;
    float4* buf[2];           // ping-pong (illumination rgb | variance); k_denoise_prep writes buf[0], level i reads buf[i & 1]
};

// The pixel's linear value exactly as k_resolve forms it (per-sub-pixel mean, clamp, mean of four), demodulated; its
// luminance variance = the sample variance of the four clamped sub-pixel means' luminances / 4.
__global__ void __launch_bounds__(DENOISE_THREADS) k_denoise_prep(DenoiseArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.width * a.height) return;
    const float4 g = a.ga[i];
    float3 px;
    float var;
    if (a.accum) {
        const int y = i / a.width, x = i - y * a.width;
        const uint32_t ks_done = a.tile_ks ? a.tile_ks[(y / TILE) * a.tiles_x + x / TILE] : a.ks_done;
        float m[4];
        px = f3(0.f, 0.f, 0.f);
        for (int s = 0; s < 4; ++s) {
            const uint32_t cnt = ks_done > (uint32_t)s ? (ks_done - (uint32_t)s + 3u) / 4u : 0u;
            const float inv = cnt ? 1.0f / (float)cnt : 0.0f;
            const float4 v = a.accum[(size_t)i * 4 + s];
            const float3 c = f3(clamp01(v.x * inv), clamp01(v.y * inv), clamp01(v.z * inv));
            px.x += c.x * 0.25f;
            px.y += c.y * 0.25f;
            px.z += c.z * 0.25f;
            m[s] = lum709(c.x, c.y, c.z);
        }
        const float mean = 0.25f * (m[0] + m[1] + m[2] + m[3]);
        var = ((m[0] - mean) * (m[0] - mean) + (m[1] - mean) * (m[1] - mean) + (m[2] - mean) * (m[2] - mean) +
               (m[3] - mean) * (m[3] - mean)) * (1.0f / 12.0f);
    } else {
        const float4 c = a.buf[1][i];
        px = f3(c.x, c.y, c.z);
        var = c.w;
    }
    a.buf[0][i] = demodulate(px, var, f3(g.x, g.y, g.z));
}

// (in / out: the level's two buffers, picked on the host — a run-time index into a.buf would put the array on the stack)
__global__ void __launch_bounds__(DENOISE_THREADS) k_atrous(DenoiseArgs a, const float4* __restrict__ in, float4* __restrict__ out,
                                                            int step, DenoiseSigmas s) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.width * a.height) return;
    const int y = i / a.width, x = i - y * a.width;
    out[i] = atrous_pixel(in, a.ga, a.gn, a.width, a.height, x, y, step, s);
}

// remodulation, then k_resolve's tail: clamp -> ^(1/2.2) * 255 + 0.5 -> `as u8`; rgb8 (scan-line) and / or the linear rgb
__global__ void __launch_bounds__(DENOISE_THREADS) k_denoise_out(DenoiseArgs a, const float4* __restrict__ in, unsigned char* __restrict__ rgb8,
                                                                 float* __restrict__ out3) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.width * a.height) return;
    const float4 g = a.ga[i];
    const float3 v = remodulate(in[i], f3(g.x, g.y, g.z));
    if (out3) {
        out3[3 * (size_t)i] = v.x;
        out3[3 * (size_t)i + 1] = v.y;
        out3[3 * (size_t)i + 2] = v.z;
    }
    if (rgb8) {
        rgb8[3 * (size_t)i] = to_u8(powf(clamp01_keep_nan(v.x), 1.0f / 2.2f) * 255.0f + 0.5f);
        rgb8[3 * (size_t)i + 1] = to_u8(powf(clamp01_keep_nan(v.y), 1.0f / 2.2f) * 255.0f + 0.5f);
        rgb8[3 * (size_t)i + 2] = to_u8(powf(clamp01_keep_nan(v.z), 1.0f / 2.2f) * 255.0f + 0.5f);
    }
}

}  // namespace rtb
