// shade_body.cuh — the body of k_shade and k_shade_metal (wavefront.cuh), #included inside each kernel's braces.  It sees the
// kernel's template parameters MODE, NP, NS, MESH, THREADS, INLINE and its parameters `a` (the __grid_constant__ RenderArgs) and
// `c`.  Kept as one text rather than a device function that both kernels call: with the call, ptxas schedules the existing
// k_shade instantiations differently; included here they compile to exactly the code they had before the metal kernels existed.
    constexpr bool FAST = MODE == 1 || MODE == 2;
    constexpr bool DIEL = MODE == 3 || MODE == 5 || MODE == 6 || MODE == 7;
    constexpr bool ALL = MODE == 4 || MODE == 5 || MODE == 7;   // RTB_EST_NEE_ALL_LIGHTS
    constexpr bool MET = MODE == 6 || MODE == 7;                // rough metal (brdf 4)
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
    const bool select_b1 = ALL ? hdr->lights_select != 0 : light_is_mesh;   // a non-Phong vertex draws block 1 for its light choice
    const bool mis = MODE == 1 || ALL || MET ? false : (MODE == 2 ? true : a.estimator == 1);     // the reference's dead "MIS" branch
    // RTB_EST_MIS_BALANCE (general instantiation only): next-event estimation and the BRDF sample combined with the balance
    // heuristic — what src/scene.rs:187 ("TODO: Do multiple importance sampling properly") asks for.  Diffuse surfaces under
    // a sphere light; Phong surfaces keep plain NEE (the reference's Phong sampler never leaves the local frame, its pdf
    // for a world direction is undefined).  Never used for parity.
    const bool mis2 = FAST || ALL ? false : a.estimator == 2;
    const bool probe_mode = FAST ? false : a.probe_px != nullptr;
    const float3 Le = f3(sh.mats[light_obj].emitted);
    const int n_prims = a.S.n_prims, n_planes = a.S.n_planes;
    const ShadowQueue& SQ = a.sqout;
    uint32_t* const ctr_front = &C->ext_head(1 - c);
    uint32_t* const ctr_back = &C->ext_tail(1 - c);
    uint32_t* const ctr_sh = &C->sh_head(1 - c);
    uint32_t n_ext = 0, n_ext_bvh = 0, n_sh = 0, n_sh_bvh = 0, n_queued = 0;   // rays of this warp: sums of its ballots
    uint32_t n_sh_inline = 0;   // INLINE: shadow / probe rays this lane traversed here (counted as BVH shadow rays, never pending)
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
    // output segments of this warp (see seg_alloc); none is reserved yet
    __shared__ ShadeSegs segs[THREADS / 32];
    ShadeSegs& W = segs[threadIdx.x >> 5];
    if (lane < 3) {
        W.base[lane] = 0;
        W.used[lane] = SHADE_SEG;
    }
    __syncwarp();
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

        // The trip runs in four phases, so that each output of the vertex dies right where it is stored: (A) divergent shading
        // produces only raw quantities, (B) the analytic pair + box test, (C) the shadow push, (D) keep / park and the path push.
        // A queue entry is put together at its store, from `pos`, the direction and the throughput; no packed copy of it stays live.
        bool ext_push = false, want_sh = false, pr_push = false, pr_try = false;
        // raw outputs of (A); each is written before it is read under the same flag
        float3 pos, nbeta;
        uint32_t pcode, eflags;   // hit's pcode; pcode + flags of the extension entry
        float3 next_dir = f3(0.f, 0.f, 0.f), sh_dir = f3(0.f, 0.f, 0.f), sh_contrib;
        float sh_tlim = 0.f;
        float4 ev = make_float4(0.f, 0.f, 0.f, 0.f);   // stale `o` of a specular vertex | pdf of a balance-heuristic BRDF sample
        float4 pd, pc;   // dead-MIS probe entry (its origin is `pos`)
        const uint32_t acc = __float_as_uint(d4.w);
        const uint32_t sdw = __float_as_uint(b4.w);

        // ---- (A) divergent shading
        if (cur_valid) {
            const uint32_t id = __float_as_uint(h2.y);
            if (id != PC_NONE) {
                const float t = h2.x;
                const float3 o = f3(o4), d = f3(d4);
                const uint32_t origin = __float_as_uint(o4.w);
                float3 beta = f3(b4);
                const uint32_t sample = sdw >> 12, depth = sdw & 0xfffu;
                const HitGeom hg = hit_geometry(sh, o, d, t, id, tri_n);
                pos = hg.pos;
                pcode = hg.pcode;
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
                    if constexpr (DIEL) {
                        if (pm.brdf != 3) beta = beta * f3(pm.k) * inv_pp;   // a dielectric vertex has put its weight into beta already
                    } else {
                        beta = beta * f3(pm.k) * inv_pp;
                    }
                } else if constexpr (ALL) {
                    // behind a diffuse or Phong vertex: its light sample has counted the emitters of the table, not the others
                    if (emits && reinterpret_cast<const int32_t*>(reinterpret_cast<const char*>(hdr) + 256 * (size_t)hdr->off_light_of)[hg.obj] < 0)
                        accum_add(a.accum, acc, beta * emitted);
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
                    float pick_u = 0.f;
                    if (!FAST && (mat.brdf == 2 || select_b1) && !(DIEL && mat.brdf == 3)) {
                        const float4 r1 = rng_block(rng_pixel, sample, depth, 1u, a.keys);
                        lobe_u = r1.x;
                        select_u = r1.y;
                        if constexpr (ALL) pick_u = r1.z;   // which entry of the light table
                    }
                    const float4 r0 = make_float4(vr.light_u1, vr.light_u2, vr.rr, select_u);
                    const float4 rb = make_float4(vr.brdf_u1, vr.brdf_u2, lobe_u, 0.f);
                    if (DIEL && mat.brdf == 3) {
                        // dielectric: reflect or refract with the Fresnel probability; the TRUE direction d, never the stale `o`.
                        // No light sample: emission reached through glass is added at the next hit (PC_SPEC_PENDING).
                        if (r0.z < p) {
                            bool refracted;
                            next_dir = dielectric_scatter(d, hg.n, (hg.pcode & PC_FLIPPED) != 0u, mat.k.y, mat.k.x, rb.x, refracted);
                            nbeta = beta * inv_p;
                            if (refracted) {
                                // the ray leaves through the other side: with the flip bit toggled the self-intersection rule sees
                                // its origin 1e-5 beyond the surface (spheres: on it, roots 0 and 2b), so the origin moves there
                                pcode = hg.pcode ^ PC_FLIPPED;
                                if (mat.geom != 0) pos = hg.pos - (2.0f * SURF_OFFSET) * hg.n;   // not a sphere
                                nbeta = nbeta * f3(mat.color_d);   // no eta^2 factor: camera and light lie outside every medium
                            }
                            ext_push = true;
                            eflags = pcode | PC_SPEC_PENDING;
                        }
                    } else if (mat.brdf == 1) {  // specular branch, src/scene.rs:170-185
                        if (r0.z < p) {
                            next_dir = flip_across(ovec, hg.n);
                            ext_push = true;
                            eflags = hg.pcode | PC_SPEC_PENDING | PC_STALE_O;
                            nbeta = beta;
                            ev = make_float4(ovec.x, ovec.y, ovec.z, 0.f);  // the recursion is handed `o`, not -i (src/scene.rs:178)
                        }
                    } else {
                        // ---- direct light
                        float3 y, ny, Le_y;   // Le_y: the sampled light's emission (ALL)
                        float pdf_a;
                        if (FAST) light_sample_sphere(a.light_sphere, a.light_pdf, r0, y, ny, pdf_a);
                        else if (ALL) light_sample_all(a.S, sh, hdr, r0, pick_u, hg.pos, y, ny, pdf_a, Le_y);
                        else light_sample<FAST>(a.S, sh.prims, hdr, r0, y, ny, pdf_a);
                        float3 dv = y - hg.pos;
                        float r2 = dot(dv, dv);
                        float inv_dist = rsqrtf(r2);
                        float dist = r2 * inv_dist;
                        float3 inc = dv * inv_dist;
                        // a metal sees the TRUE direction of arrival: the stale `o` belongs to the reference's materials only
                        float3 f = MET && mat.brdf == 4 ? metal_eval(f3(mat.color_s), mat.k.x, hg.n, -d, inc) : brdf_eval<FAST>(mat, hg.n, ovec, inc);
                        float3 contrib;
                        if (!mis) {  // live NEE, src/scene.rs:217-229 (no cosine is clamped)
                            float g = ALL ? light_weight(hg.n, ny, inc, r2, pdf_a) : __fdividef(dot(hg.n, inc) * dot(ny, -inc), r2 * pdf_a);
                            contrib = beta * (ALL ? Le_y : Le) * f * g;
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
                            want_sh = true;     // mutually_visible is resolved in (B), together with the extension ray
                            sh_dir = inc;
                            sh_tlim = dist - SHADOW_MARGIN;
                            sh_contrib = contrib;
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
                                    pr_try = true;
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
                                }
                            }
                        }
                        // ---- russian roulette + continuation, src/scene.rs:231-240
                        if (MET && mat.brdf == 4) {
                            // metal: a visible normal of the GGX lobe; weight F G2 / G1.  Not specular: no PC_SPEC_PENDING, no stale `o`
                            float3 w;
                            if (r0.z < p && metal_sample(f3(mat.color_s), mat.k.x, hg.n, -d, rb.x, rb.y, next_dir, w)) {
                                nbeta = beta * w * inv_p;
                                ext_push = true;
                                eflags = hg.pcode;
                            } else {
                                next_dir = f3(0.f, 0.f, 0.f);
                            }
                        } else if (r0.z < p) {
                            float pdf1;
                            brdf_sample<FAST>(mat, hg.n, ovec, rb, next_dir, pdf1);
                            if (next_dir.x != 0.f || next_dir.y != 0.f || next_dir.z != 0.f) {
                                if (FAST || mat.brdf == 0) nbeta = beta * f3(mat.k) * inv_p;  // f (n.i) / pdf == kd exactly
                                else nbeta = beta * brdf_eval(mat, hg.n, ovec, next_dir) * (dot(hg.n, next_dir) / (pdf1 * p));
                                ext_push = true;
                                eflags = hg.pcode;
                                if (mis2 && mat.brdf == 0) {   // the sample's pdf travels with the ray (see PC_MIS_PENDING)
                                    eflags = hg.pcode | PC_MIS_PENDING;
                                    ev = make_float4(0.f, 0.f, 0.f, pdf1);
                                }
                            }
                        }
                    }
                }
            }
        }
        // shadow rays of this trip (NEE candidates, dead-MIS probes): counted from the warp's ballots
        uint32_t trip_sh = __popc(__ballot_sync(0xffffffffu, want_sh));
        unsigned mp = 0;
        if (mis) {
            // dead-MIS probes need no pair test: pushed here, so their entries are dead before (B)
            trip_sh += __popc(__ballot_sync(0xffffffffu, pr_try));
            mp = __ballot_sync(0xffffffffu, pr_push);
            if (mp) {
                const uint32_t slot = seg_alloc<1>(W, nb, 2u, ctr_sh, mp, lane);
                if (pr_push) {
                    if (slot < a.SPcap) { SQ.o[slot] = make_float4(pos.x, pos.y, pos.z, __uint_as_float(pcode)); SQ.d[slot] = pd; SQ.c[slot] = pc; }
                    else atomicAdd(&C->overflow, 1u);
                }
                n_sh_bvh += __popc(mp);
            }
        }
        n_sh += trip_sh;

        // ---- (B) analytic half of BOTH trace_ray calls this vertex makes (extension: nearest hit; shadow: mutually_visible,
        // src/scene.rs:258-270), here where every lane does it together.  Rays that can still reach the mesh box afterwards are
        // queued for k_traverse.
        float ta;
        uint32_t ida;
        bool ext_box = false;
        if (ext_push || want_sh) {
            bool occ, sh_box;   // can the two rays still reach the mesh box?  (both at once: shared terms, packed products)
            if (NP == 8) analytic_pair_small8(a.ss, n_planes, n_prims, origin_group_of(sh, pcode), pos, pcode, next_dir, ta, ida, sh_dir, sh_tlim, occ);
            else if (NP > 0) analytic_pair_small<NP, NS>(a.ss, origin_group_of(sh, pcode), pos, pcode, next_dir, ta, ida, sh_dir, sh_tlim, occ);
            else analytic_pair(sh, n_planes, n_prims, pos, pcode, next_dir, ta, ida, sh_dir, sh_tlim, occ);
            if (MESH) ray_pair_hits_bvh_box(a.S, pos, next_dir, ta, sh_dir, sh_tlim, ext_box, sh_box);
            else ext_box = sh_box = false;   // no triangles in the scene: no ray ever leaves this kernel for k_traverse
            if (want_sh) {   // from here on: the shadow ray goes to the queue
                want_sh = false;
                if (occ) {
                } else if (sh_box && INLINE) {   // mutually_visible's mesh half, right here
                    ++n_sh_inline;
                    uint32_t idt = PC_NONE;
                    float tt = sh_tlim;
                    if (!bvh_traverse<true, false>(a.S, sh, pos, sh_dir, pcode, tt, idt, sh_tlim + SHADOW_MARGIN, nullptr)) accum_add(a.accum, acc, sh_contrib);
                } else if (sh_box) {
                    want_sh = true;
                } else {
                    accum_add(a.accum, acc, sh_contrib);
                }
            }
        }
        const bool sh_push = want_sh;

        // ---- (C) shadow push; the shadow ray's values are dead afterwards
        const unsigned ms = __ballot_sync(0xffffffffu, sh_push);
        if (ms) {
            const uint32_t slot = seg_alloc<1>(W, nb, 2u, ctr_sh, ms, lane);
            if (sh_push) {
                if (slot < a.SPcap) {
                    SQ.o[slot] = make_float4(pos.x, pos.y, pos.z, __uint_as_float(pcode));
                    SQ.d[slot] = make_float4(sh_dir.x, sh_dir.y, sh_dir.z, sh_tlim);
                    SQ.c[slot] = make_float4(sh_contrib.x, sh_contrib.y, sh_contrib.z, __uint_as_float(acc));
                } else {
                    atomicAdd(&C->overflow, 1u);
                }
            }
            n_sh_bvh += __popc(ms);
        }

        // ---- (D) extension: where does the path go?  In registers if its next hit is final and it queued no shadow ray.
        n_ext += __popc(__ballot_sync(0xffffffffu, ext_push));
        n_ext_bvh += __popc(__ballot_sync(0xffffffffu, ext_push && ext_box));
        if (INLINE && ext_push && ext_box) bvh_traverse<false, false>(a.S, sh, pos, next_dir, pcode, ta, ida, 0.f, nullptr);   // the hit is final afterwards
        const bool ext_front = !INLINE && ext_box;
        bool keep = ext_push && !ext_front && !park && (!(sh_push || pr_push) || !sh_tight);
        if (ext_push && !ext_front && ida == PC_NONE) {   // left the scene: nothing to shade
            keep = false;
            ext_push = false;
        }
        if (keep) ext_push = false;
        // slots from the warp's segments (see seg_alloc), written straight away
        const unsigned mf = __ballot_sync(0xffffffffu, ext_push && ext_front);
        const unsigned mb = __ballot_sync(0xffffffffu, ext_push && !ext_front);
        if (mf | mb) {
            uint32_t slot = 0;
            if (mf) { const uint32_t v = seg_alloc<1>(W, nb, 0u, ctr_front, mf, lane); if (ext_front) slot = v; }
            if (mb) { const uint32_t v = seg_alloc<-1>(W, nb, 1u, ctr_back, mb, lane); if (!ext_front) slot = v; }
            if (ext_push && slot >= a.Pcap) { atomicAdd(&C->overflow, 1u); ext_push = false; }
            if (ext_push) {
                N.o[slot] = make_float4(pos.x, pos.y, pos.z, __uint_as_float(eflags));
                N.d[slot] = make_float4(next_dir.x, next_dir.y, next_dir.z, __uint_as_float(acc));
                N.beta[slot] = make_float4(nbeta.x, nbeta.y, nbeta.z, __uint_as_float(sdw + 1u));   // depth + 1 (< 4096: no carry)
                N.hit[slot] = make_float2(ta, __uint_as_float(ida));
                if (eflags & (PC_STALE_O | PC_MIS_PENDING)) N.ov[slot] = ev;
            }
            n_queued += __popc(__ballot_sync(0xffffffffu, ext_push));
        }
        if (ms | mp) sh_tight = W.base[2] + SHADE_SEG > a.SP;   // warp-uniform: where this warp's current shadow segment ends
        // ---- next vertex of the same path, straight from registers
        cur_valid = keep;
        if (keep) {
            o4 = make_float4(pos.x, pos.y, pos.z, __uint_as_float(eflags));
            d4 = make_float4(next_dir.x, next_dir.y, next_dir.z, __uint_as_float(acc));
            b4 = make_float4(nbeta.x, nbeta.y, nbeta.z, __uint_as_float(sdw + 1u));
            h2 = make_float2(ta, __uint_as_float(ida));
            if (INLINE) {    // the next hit may be a triangle (traversed above): its normal, and the stale `o` in its own register
                ev_keep = ev;
                if (ida != PC_NONE && ida >= TRI_BASE) tri_n = __ldg(a.S.tri_nrm + (ida - TRI_BASE));
            } else {
                tri_n = ev;  // stale `o` of a specular vertex (PC_STALE_O in eflags); analytic hits need no triangle normal
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
        const uint32_t fu = W.used[0] & ~SEG_NEXT, bu = W.used[1] & ~SEG_NEXT, su = W.used[2] & ~SEG_NEXT;
        for (uint32_t k = fu + lane; k < SHADE_SEG; k += 32) mark_path(seg_slot<1>(W.base[0], k));
        for (uint32_t k = bu + lane; k < SHADE_SEG; k += 32) mark_path(seg_slot<-1>(W.base[1], k));
        for (uint32_t k = su + lane; k < SHADE_SEG; k += 32) mark_sh(seg_slot<1>(W.base[2], k));
        const uint32_t nf = __shfl_sync(0xffffffffu, nb, 0), nbk = __shfl_sync(0xffffffffu, nb, 1) - 1u, ns = __shfl_sync(0xffffffffu, nb, 2);
        if (W.used[0] & SEG_NEXT) for (uint32_t k = lane; k < SHADE_SEG; k += 32) mark_path(seg_slot<1>(nf, k));
        if (W.used[1] & SEG_NEXT) for (uint32_t k = lane; k < SHADE_SEG; k += 32) mark_path(seg_slot<-1>(nbk, k));
        if (W.used[2] & SEG_NEXT) for (uint32_t k = lane; k < SHADE_SEG; k += 32) mark_sh(seg_slot<1>(ns, k));
    }
    // counters (warp-uniform, but for the inline shadow rays)
    if (INLINE)
        for (int off = 16; off; off >>= 1) n_sh_inline += __shfl_down_sync(0xffffffffu, n_sh_inline, off);
    if (lane == 0) {
        if (n_queued) { atomicAdd(&C->live[1 - c], n_queued); atomicAdd(&C->paths_queued, (unsigned long long)n_queued); }
        if (n_sh_bvh) atomicAdd(&C->sh_live[1 - c], n_sh_bvh);
        if (n_ext) atomicAdd(&C->rays_extension, (unsigned long long)n_ext);
        if (n_ext_bvh) atomicAdd(&C->rays_bvh, (unsigned long long)n_ext_bvh);
        if (n_sh) atomicAdd(&C->rays_shadow, (unsigned long long)n_sh);
        if (n_sh_bvh + n_sh_inline) atomicAdd(&C->shadow_bvh, (unsigned long long)(n_sh_bvh + n_sh_inline));
    }
