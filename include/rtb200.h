/* rtb200.h — C ABI of librtb200.so, the B200-native (sm_100a) replacement for the per-pixel
 * radiance loop of SuneelFreimuth/raytracer-server.
 *
 * The reference has no FFI; its seam is three Rust signatures (citations relative to the
 * reference tree).  Each entry point below names the one it stands in for:
 *
 *   Scene::from_toml<R: Read>(&mut R) -> Result<Scene, LoadTomlError>      src/scene.rs:143-150
 *   sample_pixel(x, y, width, height, samples_per_pixel, &Scene) -> Vec3    src/server.rs:320-364
 *   RenderJob::run(&self, &Scene, width, height, spp) -> bool               src/server.rs:157-199
 *
 * Plain pointers and sizes only; no C++/torch types.  All functions return RTB_OK (0) or a
 * negative error code and set a thread-local message readable with rtb_last_error().
 * A scene handle is immutable after creation and may be shared by host threads; every render
 * call / job owns its own CUDA stream and scratch buffers.
 * There is NO CPU fallback: without a CUDA device every compute entry point fails with RTB_ECUDA.
 */
#ifndef RTB200_H
#define RTB200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RTB_ABI_VERSION 2

/* error codes — LoadTomlError::{Io,Parse,MeshLoad} (src/scene.rs:350-355) plus the reference's
 * panics turned into codes: no emitter = unreachable!() (src/scene.rs:136); plane light =
 * unimplemented!() (src/geometry.rs:593). */
enum {
    RTB_OK = 0,
    RTB_EIO = -1,
    RTB_EPARSE = -2,
    RTB_EMESH = -3,
    RTB_ENOLIGHT = -4,
    RTB_EUNSUPPORTED = -5,
    RTB_ECUDA = -6,
    RTB_EINVAL = -7,
    RTB_ESTOPPED = -8,  /* rtb_job_next* after rtb_job_cancel (the job yields nothing more) */
    RTB_ECANCELLED = 1  /* rtb_render* / rtb_job_end: RenderJob::run returns true when stopped early (src/server.rs:198) */
};

typedef struct rtb_scene rtb_scene;
typedef struct rtb_job rtb_job;

/* estimator selection (src/scene.rs:187-229) */
#define RTB_EST_NEE 0      /* live branch: next-event estimation, src/scene.rs:217-229 */
#define RTB_EST_MIS_DEAD 1 /* the `if false` "MIS" branch verbatim, src/scene.rs:189-216 */
#define RTB_EST_MIS_BALANCE 2 /* NOT in the reference: light sample + BRDF sample combined with the balance heuristic, i.e. the
                                 "TODO: Do multiple importance sampling properly" of src/scene.rs:187 done.  Same expectation as
                                 RTB_EST_NEE, less variance near the light; sphere lights only; never used for parity */
#define RTB_EST_NEE_ALL_LIGHTS 3 /* NOT in the reference: next-event estimation over EVERY emitter, not just the first.  The light
                                 table (rtb_scene_lights) holds each sphere or mesh with weight w = lum(max(emitted, 0)) * area > 0
                                 (lum = Rec. 709 weights, area after the transforms: 4 pi r^2, or a mesh's true area), in object
                                 order; a vertex picks entry i with p_i = w_i / sum w (block 1 z of the RNG contract), a triangle
                                 of a mesh light by area (block 1 y) and a uniform point (block 0 light u1, u2), and adds
                                 beta Le_i f max(n.w, 0) |n_y.w| / (r^2 p_i / area_i) if the point is visible.  Emission reached
                                 from a diffuse or Phong vertex counts only for emitters outside the table (planes, zero weight);
                                 at depth 1 and behind a mirror or glass it always counts.  With one sphere light this is
                                 RTB_EST_NEE but for its unclamped cosines. */

/* mesh acceleration (Mesh::intersect, src/geometry.rs:883-905) */
#define RTB_ACCEL_LBVH 0             /* true nearest hit = the reference's brute-force branch (:887-903), through the device-built BVH (binned SAH, linear node table) */
#define RTB_ACCEL_OCTREE_REFERENCE 1 /* the branch the reference actually runs: its per-mesh octree with the early exit on the first child
                                        that reports any hit (:1237-1295; Octree::build :1149-1216 restated on the host).  NOT a nearest-hit
                                        structure — it is what makes the Rust binary's flying_unicorn differ from the exact image by 30 dB.
                                        Slower than the LBVH; for results identical to the binary's */

/* Render request.  spp has the reference's meaning: spp/4 samples in each of 2x2 sub-pixels
 * (src/server.rs:332), so spp < 4 renders black.  (rank, world) select an interleaved tile
 * shard: this call renders the 32x32 tiles t with t % world == rank (world = 1: whole frame). */
typedef struct rtb_params {
    int32_t width;
    int32_t height;
    int32_t spp;
    int32_t estimator; /* RTB_EST_* ("use_mis" of the orphaned config.toml:5) */
    uint64_t seed;     /* Philox key; the reference is unseeded (rand::random) */
    int32_t rank;
    int32_t world;
    int32_t pool_paths; /* in-flight path slots; 0 = default */
    int32_t accel;      /* RTB_ACCEL_*: which Mesh::intersect the mesh rays get */
    int32_t tuning[4];  /* experiment knobs, 0 = library defaults: [0] 1 = counting build (bvh_node_visits / bvh_tri_tests), [1] refill
                           threshold and [2] inner steps of k_traverse, [3] coherence binning (1 off, 2..5 cell bits per axis, +256 octant-major) */
} rtb_params;

typedef struct rtb_scene_info {
    int32_t n_objects;
    int32_t n_planes;
    int32_t n_spheres;
    int32_t n_meshes;
    int32_t n_triangles;
    int32_t light_object; /* Scene::light_source, src/scene.rs:129-137 */
    int32_t bvh_nodes;
    int32_t bvh_leaves;
    int32_t device;
    int32_t bvh_depth;    /* inner-node levels on the longest root-to-leaf path; the loader refuses trees deeper than the
                             traversal stack (96) with RTB_EUNSUPPORTED */
    int32_t octree_nodes;     /* RTB_ACCEL_OCTREE_REFERENCE tables: 0 until the first request for that mode builds them */
    int32_t octree_tri_refs;  /* triangle references in the octrees' leaves (the reference copies a triangle into every octant it overlaps) */
    float bvh_min[3];
    float bvh_max[3];
    float camera_pos[3];
    float camera_dir[3];
    double build_ms; /* device LBVH build */
} rtb_scene_info;

/* one object as the loader built it (f64, after transforms) — Object / Geometry, src/scene.rs:10-15 */
typedef struct rtb_object_info {
    int32_t brdf;          /* 0 diffuse, 1 specular, 2 phong, 3 dielectric */
    int32_t geometry;      /* 0 sphere, 1 plane, 2 mesh (cube / prism / OBJ) */
    int32_t n_triangles;
    int32_t first_triangle; /* global triangle index of the mesh's first triangle, or -1 */
    double emitted[3];
    double k[3];           /* kd | ks | phong {kd, ks, power} | dielectric {ior, orientation sign, 0}: the sign is +1 when the
                              stored normals point out of the medium (sphere: radial, plane: n, mesh: see rtb_object_desc) */
    double color_d[3];
    double color_s[3];
    double pos[3];
    double n[3];
    double r;
    double bb_min[3];      /* Mesh::bounding_box incl. the scale() quirk (src/geometry.rs:503-506) */
    double bb_max[3];
    double surface_area;   /* Mesh::surface_area: computed before the transforms, never refreshed */
} rtb_object_info;

/* counters of the last finished render / job — counted on the device, never inferred */
typedef struct rtb_stats {
    uint64_t samples;        /* received_radiance calls */
    uint64_t rays_primary;   /* trace_ray calls, by kind */
    uint64_t rays_extension;
    uint64_t rays_shadow;
    uint64_t iterations;     /* wavefront iterations */
    uint64_t kernel_launches;
    uint64_t bvh_node_visits; /* only filled by counting builds (rtb_trace_* with count_work) */
    uint64_t bvh_tri_tests;
    double render_ms;        /* CUDA-event time of the whole device-side render */
    double extend_ms;        /* CUDA-event time of k_traverse (all LBVH queries: closest + any hit), summed over launches */
    double bin_ms;           /* CUDA-event time of the coherence binning in front of k_traverse (k_bin_keys / _scan / _scatter) */
    double generate_ms;
    double resolve_ms;
    double shade_ms;         /* k_shade */
    uint64_t rays_bvh;       /* primary + extension rays that needed the LBVH (the rest end at an analytic primitive) */
    uint64_t shadow_bvh;     /* shadow rays that needed the LBVH */
    uint64_t paths_queued;   /* path-queue entries k_shade wrote (a path stays in registers while its next hit is analytic) */
    double first_record_ms;  /* streaming jobs: host time from rtb_job_begin until the first record could be delivered (-1: none yet) */
    double wall_ms;          /* streaming jobs: host time from rtb_job_begin until the last worker finished (or until now) */
} rtb_stats;

/* ---- scene: Scene::from_toml + SceneSpec::to_scene (src/scene.rs:143-150, 357-441) ---------
 * Same TOML grammar and semantics: transform order, bbox-centre pivots and the scale() bbox
 * quirk (src/geometry.rs:445-510), first-emitter light rule, OBJ subset (v / f a/b/c, triangles
 * only, src/geometry.rs:777-833).  Mesh paths resolve against assets_dir (the reference uses
 * <argv[1]>/assets, src/scene.rs:405).  `device` is the CUDA ordinal that will own the scene;
 * device = -1 creates a host-only handle (loader checks on machines without a GPU): info / object /
 * triangle queries work, every compute entry point fails with RTB_ECUDA. */
int rtb_scene_load_toml(const char* toml_path, const char* assets_dir, int device, rtb_scene** out);
int rtb_scene_load_toml_string(const char* toml_text, const char* assets_dir, int device, rtb_scene** out);
void rtb_scene_destroy(rtb_scene* scene);

/* ---- programmatic scene (no TOML): the objects a host already has in memory ---------------------
 * One entry per Object (src/scene.rs:10-15).  Geometry is final (no transforms are applied):
 * sphere {pos, r}; plane {pos, n}; mesh = n_triangles x 9 floats (a, b, c per triangle, vertex order as in
 * Mesh::triangle, src/geometry.rs:872-877).  Same light rule and error codes as the TOML path. */
typedef struct rtb_object_desc {
    double emitted[3];
    int32_t brdf;           /* 0 diffuse {k = kd}, 1 specular {k = ks}, 2 phong {k = kd, ks, power; color_d; color_s},
                               3 dielectric {k = ior, 0, 0 (ior finite, > 0); color_d = transmission tint, each in [0, 1]}:
                               smooth glass, air outside.  Outside is the side of a sphere's outward normal, the side a
                               plane's n points to, and for a mesh the outside of the solid it bounds: the loader winds
                               each connected piece consistently and orients it by its signed volume (f64), and keeps
                               the stored normal norm((c-a) x (b-a)) of the first triangle, turning triangles wound
                               against it around (b <-> c).  Meant for closed meshes; an open one gets an arbitrary side. */
    int32_t geometry;       /* 0 sphere, 1 plane, 2 mesh */
    double k[3];
    double color_d[3];
    double color_s[3];
    double pos[3];
    double n[3];            /* plane normal */
    double r;               /* sphere radius */
    const float* triangles; /* mesh: n_triangles * 9 floats */
    int64_t n_triangles;
} rtb_object_desc;

typedef struct rtb_scene_desc {
    double camera_pos[3];
    double camera_dir[3];
    int32_t n_objects;
    int32_t reserved;
    const rtb_object_desc* objects;
} rtb_scene_desc;

int rtb_scene_create(const rtb_scene_desc* desc, int device, rtb_scene** out);

/* ---- scene + BVH as one blob, for the one-time broadcast of a multi-GPU job -------------------------------------------
 * rtb_scene_export writes the loaded objects (f64, after transforms) and the device-built LBVH tables, byte for byte as they
 * sit in device memory, into buf and returns the number of bytes (call with buf = NULL / cap too small to query the size).
 * rtb_scene_import rebuilds a scene handle on `device` from such a blob WITHOUT parsing TOML / OBJ or building a BVH: the
 * importing GPU traverses bit-identical tables.  A host-only handle (device = -1) exports the objects alone and the importer
 * builds its own LBVH.  (The reference's analogue is the Arc<HashMap<String, Scene>> every
 * connection shares, src/server.rs:24 — here the sharers are GPUs.) */
int64_t rtb_scene_export(rtb_scene* scene, void* buf, int64_t cap);
int rtb_scene_import(const void* buf, int64_t bytes, int device, rtb_scene** out);

int rtb_scene_get_info(const rtb_scene* scene, rtb_scene_info* info);
int rtb_scene_object(const rtb_scene* scene, int32_t index, rtb_object_info* out);
/* re-copy the flattened host scene (pinned) to the device; returns bytes copied via *bytes */
int rtb_scene_upload(rtb_scene* scene, uint64_t* bytes);
/* host-side view of the loader result, for cross-checks: triangles as 9 floats each (a,b,c) in
 * global triangle order; returns the count (call with cap = 0 to query) */
int64_t rtb_scene_triangles(const rtb_scene* scene, float* out9, int64_t cap);
/* the light table of RTB_EST_NEE_ALL_LIGHTS: per entry the object index, its selection probability and its area (f64);
 * returns the entry count and fills at most cap entries of each non-NULL array (call with cap = 0 to query).  Works on
 * host-only handles. */
int64_t rtb_scene_lights(const rtb_scene* scene, int32_t* objects, double* prob, double* area, int64_t cap);

/* Octree::build (src/geometry.rs:1149-1216) for one mesh object, on the host: counts4 = {nodes, parents, leaves, triangle
 * references}.  What RTB_ACCEL_OCTREE_REFERENCE traverses; needs no device. */
int rtb_scene_octree_stats(const rtb_scene* scene, int32_t object, int64_t* counts4);

const char* rtb_last_error(void);

/* ---- whole frame: what RenderJob::run has sent once all messages are out -------------------
 * rgb8_out: height*width*3 bytes, row 0 = top of the screen (message row y), exactly the bytes
 * of src/server.rs:187-189.  With world > 1 only this rank's tiles are written (others left
 * untouched).  `cancel` (may be NULL) is polled between wavefront iterations; returns
 * RTB_ECANCELLED if it became non-zero (src/server.rs:170, 198). */
int rtb_render(rtb_scene* scene, const rtb_params* params, uint8_t* rgb8_out, volatile int* cancel);

/* ---- adaptive sampling (not in the reference): stop rendering a 32x32 tile once its noise is below a target ----------
 * params.spp is the BUDGET.  Passes add pass_spp samples per pixel to every tile still active; pass p covers the samples
 * ks in [p * pass_spp, (p + 1) * pass_spp) of the budget frame's numbering (sample id sub * (spp/4) + k, ks = 4k + sub),
 * exactly like pass p of a progressive job with passes = spp / pass_spp.  A tile that received n samples per pixel
 * therefore holds a PREFIX of the budget frame's samples and is resolved with n (the bytes of that progressive job's
 * pass n / pass_spp - 1, up to the order of the fp32 sums).
 * Statistic, per pixel after every pass: for each sub-pixel s the pass's mean luminance
 * m_s = clamp01((lum(S_s) - lum_prev_s) / (pass_spp / 4)) (S_s = the sub-pixel's rgb sums, lum = Rec. 709 weights on
 * linear rgb), the batch value m = 0.25 * sum_s m_s, and a Welford (mean, M2) over the tile's B passes.  Error in 8-bit
 * output levels, after gamma_correct: mu = clamp01(mean), sigma = sqrt(M2 / (B - 1) / B) (standard error of the mean),
 * err = 255 * (min(mu + sigma, 1)^(1/2.2) - mu^(1/2.2)).
 * A tile stays active while it has fewer than spp samples per pixel AND (fewer than min_spp OR the max of err over its
 * in-frame pixels > target_levels).  target_levels = 0 never stops a tile early: the result is the uniform frame.
 * Decisions are not bit-reproducible: the fp32 sums depend on the order of atomics, so a tile right at the threshold may
 * get one pass more or fewer from run to run.  Whole frames only (world = 1).  Invalid options give RTB_EINVAL with a
 * message naming the field. */
typedef struct rtb_adaptive {
    float target_levels; /* stop a 32x32 tile once every pixel's estimated standard error is <= this many 8-bit output levels; 0 = never */
    int32_t pass_spp;    /* samples per pixel per pass (multiple of 4); params.spp (the budget) must be a multiple of it */
    int32_t min_spp;     /* no tile stops before this many samples per pixel (multiple of pass_spp, >= 2 passes) */
    int32_t reserved;    /* 0 */
} rtb_adaptive;
/* tile_spp / tile_error (optional): tiles_y*tiles_x entries, tile (tx, ty) at ty*tiles_x + tx — the samples per pixel the
 * tile received and its err after its last pass.  rgb8_out and `cancel` as for rtb_render. */
int rtb_render_adaptive(rtb_scene* scene, const rtb_params* params, const rtb_adaptive* opts, uint8_t* rgb8_out,
                        int32_t* tile_spp, float* tile_error, volatile int* cancel);

/* ---- denoising (not in the reference): an opt-in edge-aware filter of whole frames ------------------------------------
 * Guides (rtb_scene_gbuffer), per pixel from the four sub-pixel centre rays of rtb_trace_primary(sx, sy, 0, 0), each
 * followed through up to 8 specular (BRDF 1) vertices in the direction the renderer takes there (the stale-`o` quirk of
 * src/scene.rs:178 included): albedo = mean over the rays of the first non-specular hit's albedo (diffuse k, Phong
 * kd * color_d + ks * color_s) times ks of every mirror on the way, 1 for an emitter, a miss or an unfinished chain;
 * normal = the renormalised mean of the hit normals facing the ray (0 for misses); depth = mean path length to the
 * first non-specular hit over the rays that hit; obj = the object most of the four rays end on (ties: lowest sub-pixel,
 * -1 = miss).  No RNG, independent of spp: a job computes them once.
 * Filter: the pixel's linear value px exactly as the resolve forms it (per-sub-pixel clamp, mean of four) is demodulated,
 * I = px / max(albedo, 1e-3); its luminance variance is the sample variance of the four clamped sub-pixel means' Rec. 709
 * luminances / 4, divided by lum(max(albedo, 1e-3))^2.  Then `levels` a-trous levels (Dammertz et al. 2010; step 2^i at
 * level i, 5x5 B3-spline taps 1/16 1/4 3/8 1/4 1/16), each tap q of pixel p weighted by
 *     [obj_p == obj_q] * max(0, n_p . n_q)^sigma_normal * exp(-|z_p - z_q| / (sigma_depth * |grad z_p . (p - q)| + 1e-3))
 *     * exp(-|l_p - l_q| / (sigma_color * sqrt(var_p) + 1e-4))
 * (the centre tap with weight 1; l = Rec. 709 luminance of I; var_p = 3x3 Gaussian of the level's variance around p;
 * grad z by central differences), the variance carried as sum w^2 var / (sum w)^2 (SVGF, Schied et al. 2017).  The
 * result is multiplied by max(albedo, 1e-3) again and goes through the resolve's clamp, gamma and `as u8`.  No atomics:
 * the filter is deterministic for given inputs.  Whole frames only (world = 1).  Invalid options give RTB_EINVAL with a
 * message naming the field. */
typedef struct rtb_denoise {
    int32_t levels;       /* a-trous levels 1..8 (step 2^i); 0 = no filtering (the resolve through the denoise path) */
    float sigma_color;    /* luminance edge-stop, in standard deviations */
    float sigma_normal;   /* exponent of the normal edge-stop */
    float sigma_depth;    /* depth edge-stop, in units of the local depth gradient */
    int32_t reserved[4];  /* 0 */
} rtb_denoise;
/* rtb_render (adaptive = NULL) or rtb_render_adaptive with every frame denoised; tile_spp / tile_error as for
 * rtb_render_adaptive (ignored without `adaptive`) */
int rtb_render_denoised(rtb_scene* scene, const rtb_params* params, const rtb_adaptive* adaptive, const rtb_denoise* denoise,
                        uint8_t* rgb8_out, int32_t* tile_spp, float* tile_error, volatile int* cancel);
/* progressive (passes > 1) or adaptive job whose every published frame is denoised; passes = 1 renders one band */
int rtb_job_begin_denoised(rtb_scene* scene, const rtb_params* params, int32_t passes, const rtb_adaptive* adaptive,
                           const rtb_denoise* denoise, rtb_job** out);
/* the guides above for a width x height frame under RTB_ACCEL_* `accel`; row 0 = top; any output may be NULL */
int rtb_scene_gbuffer(rtb_scene* scene, int32_t width, int32_t height, int32_t accel, float* albedo3, float* normal3, float* depth,
                      int32_t* obj);
/* the filter alone on host buffers (scan-line order): linear colour, its luminance variance and the guides -> the denoised
 * linear colour (before clamp and gamma).  For tests and for callers who denoise their own images. */
int rtb_denoise_image(int device, int32_t width, int32_t height, const rtb_denoise* denoise, const float* color3,
                      const float* variance, const float* albedo3, const float* normal3, const float* depth, const int32_t* obj,
                      float* out3);

/* device-resident variants (bench `value`, multi-GPU gather): the result stays in device memory
 * owned by the caller.  d_rgb8_tiles receives this rank's pixels in tile order
 * (rtb_local_pixels() * 3 bytes); d_subpixel_sums (optional) receives the fp32 sums of the four
 * sub-pixels as float4 {r,g,b,0} per (pixel, sub-pixel), same order.  Synchronous on return. */
int64_t rtb_local_pixels(const rtb_params* params);
/* host-side tile order: (x, y) of every local pixel slot of shard (rank, world), -1/-1 for slots of
 * partial tiles that fall outside the frame; returns the slot count.  Pure CPU (no device needed). */
int64_t rtb_tile_map(const rtb_params* params, int32_t* xy, int64_t cap);
int rtb_render_device(rtb_scene* scene, const rtb_params* params, void* d_rgb8_tiles, void* d_subpixel_sums,
                      volatile int* cancel);
/* scatter `world` tile-ordered shards (concatenated, each rtb_local_pixels(rank r)*3 bytes padded
 * to shard_stride bytes) into a scan-line frame; all pointers are device pointers */
int rtb_untile_device(const rtb_params* params, const void* d_shards, int64_t shard_stride, void* d_rgb8_frame,
                      int device);
/* same, enqueued on the caller's stream (a cudaStream_t; NULL = legacy default stream) without any synchronisation */
int rtb_untile_device_async(const rtb_params* params, const void* d_shards, int64_t shard_stride, void* d_rgb8_frame,
                            int device, void* cuda_stream);

/* counters of the calling thread's most recent rtb_render* / rtb_sample_* call on this scene; a thread that has not rendered on
 * it gets the scene's most recently finished render or job (whichever thread ran it).  Jobs: rtb_job_stats. */
int rtb_get_stats(const rtb_scene* scene, rtb_stats* stats);

/* ---- streaming job: the message loop of RenderJob::run (src/server.rs:166-194) -------------
 * rtb_job_next yields records in the reference's wire shape: screen column x, screen row y
 * (top-down), n <= 60 pixels, n*3 bytes of rgb.  Returns 1 while records remain, 0 when the
 * frame is complete, RTB_ESTOPPED after rtb_job_cancel.  Records become available WHILE the frame is
 * still rendering: the frame is rendered in bands of tile rows, top-down, and each finished band is
 * resolved and copied to pinned host memory on a side stream (large frames; a frame of less than ~32 M
 * samples is one band).  Progressive mode (passes > 1, not in the reference) re-sends every record once
 * per pass with the running estimate; pass n + 1 renders while pass n is copied and consumed.
 * One consumer thread per job. */
int rtb_job_begin(rtb_scene* scene, const rtb_params* params, int32_t passes, rtb_job** out);
/* adaptive form (see rtb_adaptive): a progressive job whose tiles stop once converged.  Every pass re-sends the whole frame
 * like progressive mode; at most spp / pass_spp passes, and the job is complete (not cancelled) as soon as no tile is left
 * active, which may be earlier. */
int rtb_job_begin_adaptive(rtb_scene* scene, const rtb_params* params, const rtb_adaptive* opts, rtb_job** out);
int rtb_job_next(rtb_job* job, uint16_t* x, uint16_t* y, uint8_t* n, uint8_t* rgb /* >= 180 bytes */);
/* bulk form: up to max_records records packed exactly like the reference's binary messages,
 * [0]=0 type, [1]=n, [2..4]=x u16le, [4..6]=y u16le, then n*(r,g,b) (src/server.rs:173-190);
 * each record occupies 6+3n bytes back to back.  Returns the number of records written (0 = complete,
 * RTB_ESTOPPED = cancelled and nothing written). */
int rtb_job_next_messages(rtb_job* job, uint8_t* buf, int64_t buf_bytes, int32_t max_records, int64_t* bytes_written);
/* whole-frame form (progressive display): copies the latest finished pass (height*width*3 bytes, row 0 = top)
 * and its 0-based pass index; 1 = frame copied, 0 = all passes delivered, RTB_ESTOPPED after a cancel */
int rtb_job_next_frame(rtb_job* job, uint8_t* rgb8_out, int32_t* pass_index);
/* counters of the job so far (finished bands / passes), incl. first_record_ms / wall_ms; callable at any time before rtb_job_end */
int rtb_job_stats(rtb_job* job, rtb_stats* stats);
int rtb_job_cancel(rtb_job* job);
int rtb_job_end(rtb_job* job);

/* ---- parity hooks (no RNG) ------------------------------------------------------------------
 * Scene::trace_ray (src/scene.rs:272-289) on explicit rays.  obj = object index or -1, tri =
 * triangle index inside that object's mesh or -1, t = hit distance.  rtb_trace_primary builds the
 * camera rays of src/server.rs:353-357 for every pixel (row 0 = top) at a fixed sub-pixel
 * (sx, sy) and jitter (dx, dy).  work2 (optional) receives {bvh node visits, triangle tests}. */
int rtb_trace_primary(rtb_scene* scene, int32_t width, int32_t height, int32_t sx, int32_t sy, float dx, float dy,
                      int32_t* obj, int32_t* tri, float* t);
int rtb_trace_rays(rtb_scene* scene, int64_t n, const float* org3, const float* dir3, int32_t* obj, int32_t* tri,
                   float* t, uint64_t* work2);
/* rtb_trace_rays under a chosen RTB_ACCEL_* mode: with RTB_ACCEL_OCTREE_REFERENCE the (object, triangle, t) the reference's
 * Octree::intersect returns, which need not be the nearest triangle (src/geometry.rs:1263-1273) */
int rtb_trace_rays_accel(rtb_scene* scene, int32_t accel, int64_t n, const float* org3, const float* dir3, int32_t* obj, int32_t* tri,
                         float* t);
/* radiance of explicit (pixel x, screen row y, sample index) camera paths, fp32 rgb — the
 * path-level probe matching the oracle's or_sample_radiance under the shared RNG contract */
int rtb_sample_radiance(rtb_scene* scene, const rtb_params* params, int64_t n, const int32_t* px, const int32_t* py,
                        const int32_t* sample_idx, float* rgb3);

/* sample_pixel (src/server.rs:320-364) for a list of n pixels (x, screen row y): the Vec3 the reference's function returns
 * per pixel — all spp samples, per-sub-pixel clamp, gamma, scaled to 0..255.5, BEFORE the `as u8` of RenderJob::run —
 * as 3 floats each.  Same random numbers as the frame render, so trunc(rgb3) equals the frame's bytes up to the
 * order of the fp32 accumulation. */
int rtb_sample_pixels(rtb_scene* scene, const rtb_params* params, int64_t n, const int32_t* px, const int32_t* py, float* rgb3);

/* FP32 FMA-chain microbenchmark on `device`: measured non-tensor FP32 peak (TFLOP/s) */
int rtb_fp32_peak(int device, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* RTB200_H */
