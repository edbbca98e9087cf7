// tcrt_render_grid.cu — the render kernel for scenes whose spheres sit in a uniform grid (tcrt_build_sphere_grid; BASELINE
// configs 3 and 4: lattices of 1024 / 256 spheres).  Same contract as tcrt_render.cu (same reference functions replaced,
// same arithmetic, bit-identical results, same persistent-warp pixel queue); what differs:
//   * spheres are found with a 3D-DDA through the grid (a step costs a third of a BVH node, a ray meets a sphere after a
//     few cells), the BVH remains for rays whose origin is so far away that the reference's rounding accepts wide misses
//     (grid_margin / grid_k2_max, tcrt_render_common.cuh).  A cell is a 32-byte record that carries its first sphere's
//     geometry (an unhittable sphere when the cell is empty): the sphere test of the usual one-sphere cell starts after
//     one round of loads instead of three dependent ones (cell -> item -> sphere);
//   * ONE walk in the kernel.  A bounce needs three walks — the nearest hit of the ray, then one shadow ray per light —
//     and the megakernel inlines a nearest-hit and an any-hit walk; with the grid's code next to the BVH fallback that made
//     a bounce's instruction footprint larger than the 32 KB instruction cache (76 % hit rate, 40 % of the stall samples
//     "no instruction", 38 % fewer instructions for 14 % less time).  Here a bounce is a loop over PASSES — pass 0 the
//     ray, pass l the shadow ray to light l-1 — around a single walk whose flavour (nearest / any hit) is a warp-uniform
//     run-time flag; hit record and light arithmetic hang off the pass number.  The second and third pass find the walk
//     in the cache.
// Citations: calculatePixel RayTracer.cpp:448-638, getCollision :50-89, inShade :709-771, cosineShade :654-701,
// CollisionObject ctor SceneObject.h:47-105, SceneSphere::collision SceneSphere.cpp:50-168.
#include "tcrt_render_common.cuh"

namespace {

#ifndef TCRT_GRID_MIN_BLOCKS
#define TCRT_GRID_MIN_BLOCKS 4
#endif
#ifndef TCRT_GRID_BLOCK
#define TCRT_GRID_BLOCK 256
#endif
constexpr int kGridBlock = TCRT_GRID_BLOCK;
constexpr int kGridMinBlocks = TCRT_GRID_MIN_BLOCKS;      // the walk waits on cell and sphere loads: 4 CTAs/SM at 64 registers
// Lane::level packs, so that dead paths (DESIGN.md §4.1c) cost no register: bits 0-7 the recursion level, bits 8-16 the
// level records stacked when the path died, bits 20-22 the channels that have met a zero object colour on a stacked
// level.  A path with all three is dead: nothing of its level or any deeper one can reach the pixel.
constexpr int kLevelMask = 0xff;
constexpr int kRecShift = 8;
constexpr int kRecMask = 0x1ff;
constexpr int kZeroShift = 20;
constexpr int kDead = 7 << kZeroShift;
static_assert(TCRT_MAX_DEPTH < kLevelMask, "levels and level records have to fit their fields");

// The kernel body.  MODE kModeBand: the pixels of the band (render_grid_kernel); kModeList: the samples of a pixel list
// (render_grid_list_kernel, adaptive frames; RenderLaunch::list); kModeRays: the caller's rays (render_grid_rays_kernel,
// ray batches; RenderLaunch::ray_*); kModeViews: the pixels of a band of stacked views (render_grid_views_kernel,
// multi-view frames; RenderLaunch::view_cams).  Only the refill block, the output slot and the invalid-ray count differ.
template <int CAP, int FM, int MODE>
__device__ __forceinline__ void render_grid_body(const RenderLaunch& rl) {
    extern __shared__ float4 smem4[];
    const DeviceScene& sc = rl.scene;
    // ---- stage the sweep blob (the grid-covered spheres in front of stage_off stay in global memory) ----------------
    const int stage_off = sc.stage_off;
    const int n_stage = sc.blob_f4 - stage_off;
    for (int i = threadIdx.x; i < n_stage; i += kGridBlock) smem4[i] = __ldg(sc.blob + stage_off + i);
    __syncthreads();
    Sm sm;
    const float4* base = smem4 - stage_off;
    sm.sph = base;
    sm.fin = base + sc.fin_off;
    sm.inf = base + sc.inf_off;
    sm.light = base + sc.light_off;
    sm.clu = base + sc.clu_off;
    sm.cslot = reinterpret_cast<const int*>(base + sc.cslot_off);
    sm.idx = reinterpret_cast<const int*>(base + sc.idx_off);

    const unsigned lane = threadIdx.x & 31u;
    const unsigned lt_mask = (1u << lane) - 1u;
    const unsigned total = (MODE == kModeList || MODE == kModeRays) ? (unsigned)rl.list_n
                                                                   : (unsigned)(rl.x1 - rl.x0) * (unsigned)rl.height;
    const V3 null_color = mk(rl.null_r, rl.null_g, rl.null_b);

    float stack[CAP * 7];   // per level: local rgb, k, object rgb (local memory, touched only on reflective hits)
#ifdef TCRT_CHECKED
    for (int i = 0; i < CAP * 7; ++i) stack[i] = __uint_as_float(0x7fc0dead);
#endif
    Lane ln;
    ln.pix = -1;
    ln.level = 0;
    ln.O = mk(0.f, 0.f, 0.f);
    ln.D = mk(1.f, 0.f, 0.f);
    unsigned n_primary = 0, n_shadow = 0, n_reflect = 0;
    unsigned n_invalid = 0;        // ray mode: rays refused by the validity rule
    unsigned wcur = 0, wend = 0;   // the warp's claimed tile of pixel ids
    bool exhausted = false;

    for (;;) {
        // ---- refill: a warp that has finished its tile takes the next one (tcrt_render.cu explains the threshold) ------
        unsigned idle = __ballot_sync(kFull, ln.pix < 0);
        while (__popc(idle) >= rl.refill_min && !exhausted) {
            if (wcur == wend) {
                unsigned qb = 0;
                if (lane == 0) qb = atomicAdd(rl.queue, 32u);
                qb = __shfl_sync(kFull, qb, 0);
                if (qb >= total) {
                    exhausted = true;
                    break;
                }
                wcur = qb;
                wend = min(qb + 32u, total);
            }
            const unsigned avail = wend - wcur;
            const unsigned rank = __popc(idle & lt_mask);
            bool refused = false;
            if (ln.pix < 0 && rank < avail) {
                TCRT_CHECK(wcur + rank < total, kChkQueue);
                if (MODE == kModeRays) {
                    // the caller's ray; an invalid one gets the NaN marker and leaves the lane idle for the next ray
                    const int q = (int)(wcur + rank);
                    if (ray_from_batch(rl, q, ln.O, ln.D)) {
                        ln.pix = q;
                        ln.level = 0;
                    } else {
                        float* o = rl.out + 3 * (size_t)q;
                        o[0] = o[1] = o[2] = __uint_as_float(0x7fc00000u);
                        refused = true;
                    }
                } else {
                    int xc, z;
                    if (MODE == kModeList) list_to_sample(rl, (int)(wcur + rank), xc, z);
                    else queue_to_pixel(rl, (int)(wcur + rank), xc, z);
                    ln.pix = MODE == kModeList ? (int)(wcur + rank) : xc * rl.height + z;
                    ln.level = 0;
                    if (MODE == kModeViews) view_ray(rl, xc, z, ln.O, ln.D);
                    else primary_ray(rl, xc, z, ln.O, ln.D);
                }
            }
            if (MODE == kModeRays) {
                const unsigned n_refused = (unsigned)__popc(__ballot_sync(kFull, refused));
                n_primary -= n_refused;
                n_invalid += n_refused;
            }
            n_primary += min((unsigned)__popc(idle), avail);
            wcur += min((unsigned)__popc(idle), avail);
            idle = __ballot_sync(kFull, ln.pix < 0);
        }
        if (idle == kFull) break;
        const bool active = ln.pix >= 0;
        const bool dead = ln.level >= kDead;   // traced for the reference's ray counts only: no shading, no record

        // ---- one bounce = passes around ONE walk: pass 0 the ray, pass l the shadow ray to light l - 1 ---------------------
        V3 P = ln.O, n2 = mk(0.f, 0.f, 1.f), N = n2, refl = ln.D, color = null_color;
        float diffuse = 0.f, specular = 0.f, kref = 0.f, inten = 0.f;
        bool is_light = false, hit = false, shade = false;
        V3 local = mk(0.f, 0.f, 0.f);
#ifdef TCRT_LANE_STATS
        int st_prev = 0, st_sum = 0, st_maxsum = 0;
#endif
#pragma unroll 1
        for (int pass = 0; pass <= sc.n_lights; ++pass) {
            const bool any = pass > 0;                    // warp-uniform: nearest-hit or any-hit walk
            if (any && !__any_sync(kFull, shade)) break;  // no lane has a hit to light
            // ---- the ray of this pass --------------------------------------------------------------------------------
            V3 rO = ln.O, rD = ln.D;
            float best = rl.far_dist;    // nearest: best distance so far; shadow: distance to the light
            bool want = active;
            if (any) {
                const float4 lp = sm.light[2 * (pass - 1)];
                // inShade (:743-752): dir = L - P, |dir|, Ray(P, dir) normalises with the same length
                const V3 dir = xyz(lp) - P;
                best = __fsqrt_rn(dir.x * dir.x + dir.y * dir.y + dir.z * dir.z);
                rO = P;
                rD = div3(dir, best);
                want = shade;
                if (rl.shadows_on) {
                    // The answer only matters if this light can change `local`: a positive cosine term, the clamp of
                    // cosineShade (which runs for every unshadowed light once local > 1), or a positive specular dot
                    // product.  Otherwise the ray is counted (the reference casts it) but not traced.
                    const float c_pre = dot(n2, rD);
                    const float d_pre = dot(ln.D, rD - scale(N, 2.0f * dot(rD, N)));
                    want = shade && ((d_pre > 0.0f) || (diffuse > 0.0f && (c_pre > 0.0f || local.x > 1.0f || local.y > 1.0f || local.z > 1.0f)));
                } else {
                    want = false;        // SHADOWS_ON false: nothing is in shade
                }
            }
            // ---- the walk: linearly swept rest of the scene, then the grid (or the BVH for far origins) ----------------------
            int bkey = -1;
            bool found = false;
            if (__any_sync(kFull, want)) {
                if (want) task_linear<FM>(sm, sc, rO, rD, !any, best, bkey, found);
                bool walking = want && !found;
                // far origin: fatten().m > grid_margin, as a bound on fatten's k2 (no square root; NaN counts as far)
                const V3 dc = mk(rO.x - sc.bvh_cx, rO.y - sc.bvh_cy, rO.z - sc.bvh_cz);
                const bool far_origin = walking && !(2.0f * (dot(dc, dc) + sc.bvh_r2) <= sc.grid_k2_max);
                if (__any_sync(kFull, far_origin)) {
                    if (any ? bvh_fallback<true>(sc.bvh_sph, sc.bvh_sph_root, sm, sc, rO, rD, far_origin, &best, &bkey)
                            : bvh_fallback<false>(sc.bvh_sph, sc.bvh_sph_root, sm, sc, rO, rD, far_origin, &best, &bkey))
                        found = true;
                }
                walking = walking && !far_origin;
                // entry: slab test against the grid's box (2 * reg_margin larger than any registered box on every side)
                const float ix = rcp_approx(fabsf(rD.x) < 1e-30f ? copysignf(1e-30f, rD.x) : rD.x);
                const float iy = rcp_approx(fabsf(rD.y) < 1e-30f ? copysignf(1e-30f, rD.y) : rD.y);
                const float iz = rcp_approx(fabsf(rD.z) < 1e-30f ? copysignf(1e-30f, rD.z) : rD.z);
                const float ax = (sc.grid_lo[0] - rO.x) * ix, bx = (sc.grid_hi[0] - rO.x) * ix;
                const float ay = (sc.grid_lo[1] - rO.y) * iy, by = (sc.grid_hi[1] - rO.y) * iy;
                const float az = (sc.grid_lo[2] - rO.z) * iz, bz = (sc.grid_hi[2] - rO.z) * iz;
                const float tn = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fminf(az, bz));
                const float tf = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fmaxf(az, bz));
                const float t0 = fmaxf(tn, 0.0f);
                // a far_dist <= 0 (or NaN) still lets a sphere around the origin win with its negative distance: that
                // sphere is registered in the origin's cell, the first one visited, and the exit test stops after it
                walking = walking && (tf >= t0) && (t0 <= fmaxf(best, 0.0f));
                int cx = 0, cy = 0, cz = 0;
                float tmx = 0.f, tmy = 0.f, tmz = 0.f;
                const float dtx = sc.grid_cell[0] * fabsf(ix), dty = sc.grid_cell[1] * fabsf(iy), dtz = sc.grid_cell[2] * fabsf(iz);
                const int sx = rD.x >= 0.0f ? 1 : -1, sy = rD.y >= 0.0f ? 1 : -1, sz = rD.z >= 0.0f ? 1 : -1;
                if (walking) {
                    const float px = rO.x + rD.x * t0, py = rO.y + rD.y * t0, pz = rO.z + rD.z * t0;
                    cx = min(sc.grid_dims[0] - 1, max(0, (int)floorf((px - sc.grid_lo[0]) * sc.grid_inv_cell[0])));
                    cy = min(sc.grid_dims[1] - 1, max(0, (int)floorf((py - sc.grid_lo[1]) * sc.grid_inv_cell[1])));
                    cz = min(sc.grid_dims[2] - 1, max(0, (int)floorf((pz - sc.grid_lo[2]) * sc.grid_inv_cell[2])));
                    tmx = (sc.grid_lo[0] + sc.grid_cell[0] * (float)(cx + (sx > 0 ? 1 : 0)) - rO.x) * ix;
                    tmy = (sc.grid_lo[1] + sc.grid_cell[1] * (float)(cy + (sy > 0 ? 1 : 0)) - rO.y) * iy;
                    tmz = (sc.grid_lo[2] + sc.grid_cell[2] * (float)(cz + (sz > 0 ? 1 : 0)) - rO.z) * iz;
                }
                // stop once the cell ends beyond `lim`: the light (shadow pass), or the best hit, which then lies inside the
                // part of the ray already visited; the 2e-4 relative + absolute slack is 100x the DDA's own rounding
                // (DESIGN.md §4.5).  A lane that has stopped waits at the loop's reconvergence point.
#ifdef TCRT_LANE_STATS
                int st_len = 0;
#endif
                while (walking) {
#ifdef TCRT_LANE_STATS
                    ++st_len;
#endif
                    const int c = cx + sc.grid_dims[0] * (cy + sc.grid_dims[1] * cz);
                    TCRT_CHECK(c >= 0 && c < sc.grid_dims[0] * sc.grid_dims[1] * sc.grid_dims[2], kChkNode);
                    // the cell's record carries its first sphere (an empty cell one that no ray can hit): the test starts on
                    // ONE round of loads, the second half of the record is needed on a hit and for the cell's other spheres
                    const float4* rec = reinterpret_cast<const float4*>(reinterpret_cast<const char*>(sc.grid_cells) + 32u * (unsigned)c);
                    float4 g = __ldg(rec);
                    const float4 meta = __ldg(rec + 1);
                    int more = __float_as_int(meta.x), i = __float_as_int(meta.y), j = __float_as_int(meta.z);
                    TCRT_UNROLL_LOOP
                    for (;;) {
                        TCRT_CHECK(i >= 0 && i < sc.n_sph_bvh, kChkLeaf);
                        task_sphere(sm, g, i, rO, rD, !any, best, bkey, found);
                        if (more <= 0) break;
                        --more;
                        i = __ldg(sc.grid_items + j++);
                        g = __ldg(sc.blob + i);
                    }
                    const float t_out = fminf(fminf(tmx, tmy), tmz);
                    if (found || t_out > best * 1.0002f + 2e-4f) {
                        walking = false;
                    } else if (tmx <= tmy && tmx <= tmz) {
                        cx += sx;
                        tmx += dtx;
                        walking = (unsigned)cx < (unsigned)sc.grid_dims[0];
                    } else if (tmy <= tmz) {
                        cy += sy;
                        tmy += dty;
                        walking = (unsigned)cy < (unsigned)sc.grid_dims[1];
                    } else {
                        cz += sz;
                        tmz += dtz;
                        walking = (unsigned)cz < (unsigned)sc.grid_dims[2];
                    }
                }
#ifdef TCRT_LANE_STATS
                {   // slots: 0/1 nearest walks (warp steps, lane steps); 2/3 shadow walks; 4/5 per bounce: sum of the shadow
                    // passes' longest walks / longest per-lane SUM of shadow walks (what fusing the passes would take)
                    const int mx = __reduce_max_sync(kFull, st_len), tot = __reduce_add_sync(kFull, st_len);
                    if (lane == 0) {
                        atomicAdd(&g_lane_stats[any ? 2 : 0], (unsigned long long)mx);
                        atomicAdd(&g_lane_stats[any ? 3 : 1], (unsigned long long)tot);
                    }
                    if (any) {
                        st_prev += st_len;
                        st_sum += mx;
                        st_maxsum = __reduce_max_sync(kFull, st_prev);
                    }
                }
#endif
            }
            if (!any) {
                // ---- winner's hit record (CollisionObject ctor, SceneObject.h:47-105) ----------------------------------------
                hit = active && bkey >= 0;
                if (hit) {
                    TCRT_CHECK(bkey < sc.n_sph + sc.n_fin + sc.n_inf, kChkPrimKey);
                    const int obj = sm.idx[bkey];
                    TCRT_CHECK(obj >= 0 && obj < rl.n_objects, kChkObject);
                    const float4 surf = __ldg(sc.obj_surface + obj);
                    const float4 mat = __ldg(sc.obj_material + obj);
                    const int flags = __float_as_int(mat.w);   // bit31 light, low bits texture id + 1
                    color = xyz(surf);
                    diffuse = surf.w;
                    specular = mat.x;
                    kref = mat.y;
                    inten = mat.z;
                    is_light = flags < 0;
                    const int tex = dead ? -1 : (flags & 0x7fffffff) - 1;   // a dead level's colour is not used
                    V3 n1;
                    const V3 Pp = scale(ln.D, best) + ln.O;   // t*D + O  (SceneSphere.cpp:122, SceneFinitePlane.cpp:108)
                    if (bkey < sc.n_sph) {
                        P = Pp;
                        const float4 sg = (bkey < stage_off) ? __ldg(sc.blob + bkey) : sm.sph[bkey];
                        // n1 = normalize(P - C) (SceneSphere.cpp:129-130); n2 = normalize(n1): Ray(point, normal)
                        // re-normalises (Ray.h:21-25); N = normalize(n2): the specular term's N (:565-566)
                        n1 = normalize(Pp - xyz(sg));
                        n2 = normalize(n1);
                        N = normalize(n2);
                    } else {
                        float den;
                        float px = 0.f, py = 0.f;
                        if (FM != 0 && bkey < sc.n_sph + sc.n_fin) {
                            const float4* g = sm.fin + 4 * (bkey - sc.n_sph);
                            den = dot(ln.D, xyz(g[0]));
                            if (tex >= 0) {   // x, y of SceneFinitePlane.cpp:116-120, recomputed for the winner
                                V3 PO = Pp - xyz(g[3]);
                                px = dot(PO, xyz(g[1]));
                                py = dot(PO, xyz(g[2]));
                            }
                        } else {
                            const int slot = bkey - sc.n_sph - sc.n_fin;
                            den = dot(ln.D, xyz(sm.inf[slot]));
                            if (tex >= 0) {   // SceneInfinitePlane.cpp:59-74
                                V3 PO = Pp - xyz(__ldg(sc.inf_frame + 3 * slot + 2));
                                px = dot(PO, xyz(__ldg(sc.inf_frame + 3 * slot + 0)));
                                py = dot(PO, xyz(__ldg(sc.inf_frame + 3 * slot + 1)));
                            }
                        }
                        if (tex >= 0) color = checker(__ldg(sc.textures + 2 * tex), __ldg(sc.textures + 2 * tex + 1), px, py);
                        // computeNormal + the two re-normalisations of the plane side, tabulated at upload
                        const float4* nt = sc.obj_normals + 6 * obj + (den < 0.0f ? 0 : 3);
                        n1 = xyz(__ldg(nt));
                        n2 = xyz(__ldg(nt + 1));
                        N = xyz(__ldg(nt + 2));
                        P = Pp + scale(n1, 0.0010000000475f);   // + temp_normal * INTERSECTION_OFFSET_DIST
                    }
                    if (kref > 0.0f && !is_light) {
                        float ndi = dot(n1, ln.D);     // SceneObject.h:63
                        // -2*normal.k * n_dot_incoming + incoming.k  (SceneObject.h:81-83), then Ray() normalises
                        refl = normalize(mk(-2.0f * n1.x * ndi + ln.D.x, -2.0f * n1.y * ndi + ln.D.y, -2.0f * n1.z * ndi + ln.D.z));
                    }
                }
                // the reference casts a shadow ray per light from every non-light hit; the light passes trace the ones
                // that can change the pixel, and a warp without a live lane to shade skips them altogether
                if (rl.shadows_on) n_shadow += (unsigned)sc.n_lights * (unsigned)__popc(__ballot_sync(kFull, hit && !is_light));
#ifdef TCRT_LANE_STATS
                {   // light passes dropped at dead levels: slot 6 warp-passes skipped whole (no live lane left to shade),
                    // slot 7 lane-passes (shadow rays counted, not traced)
                    const unsigned dead_shade = __ballot_sync(kFull, hit && !is_light && dead);
                    const bool none_live = !__any_sync(kFull, hit && !is_light && !dead);
                    if (lane == 0 && rl.shadows_on && dead_shade != 0u) {
                        if (none_live) atomicAdd(&g_lane_stats[6], (unsigned long long)sc.n_lights);
                        atomicAdd(&g_lane_stats[7], (unsigned long long)__popc(dead_shade) * (unsigned long long)sc.n_lights);
                    }
                }
#endif
                shade = hit && !is_light && !dead;
            } else if (shade && (!rl.shadows_on || (want && !found))) {
                // ---- light pass - 1 reaches the hit (RayTracer.cpp:548-588); rD is the light ray ---------------------------------
                // (a light whose answer did not matter adds nothing and leaves `local` as it is: skipping it is exact)
                // intensity and colour are read here, not before the walk: nothing to keep in registers across it
                const float4 lp = sm.light[2 * (pass - 1)];
                const float4 lc = sm.light[2 * (pass - 1) + 1];
                if (diffuse > 0.0f) {        // cosineShade (:654-701)
                    const float c = dot(n2, rD);
                    if (c > 0.0f) {
                        float f = c * diffuse * lp.w;
                        local.x += f * color.x * lc.x;
                        local.y += f * color.y * lc.y;
                        local.z += f * color.z * lc.z;
                    }
                    local.x = (local.x > 1.0f) ? 1.0f : local.x;
                    local.y = (local.y > 1.0f) ? 1.0f : local.y;
                    local.z = (local.z > 1.0f) ? 1.0f : local.z;
                }
                // specular (:561-588): R = L - 2.0f*L.dot(N)*N ; (V.R)^20 by 19 multiplies
                const float two_ln = 2.0f * dot(rD, N);
                const V3 R = rD - scale(N, two_ln);
                const float d = dot(ln.D, R);
                if (d > 0.0f) {
                    float pw = d;
#pragma unroll
                    for (int i = 0; i < 19; ++i) pw *= d;
                    float s = pw * specular;
                    local.x += lc.x * s;
                    local.y += lc.y * s;
                    local.z += lc.z * s;
                }
            }
        }

#ifdef TCRT_LANE_STATS
        if (lane == 0) {
            atomicAdd(&g_lane_stats[4], (unsigned long long)st_sum);
            atomicAdd(&g_lane_stats[5], (unsigned long long)st_maxsum);
        }
#endif
        // ---- continue or finish the path --------------------------------------------------------
        bool reflected = false;
        if (active) {
            V3 tail;
            bool done = true;
            // every level below this one stacked a record, up to the one where the path died
            int n_stacked = dead ? (ln.level >> kRecShift) & kRecMask : ln.level & kLevelMask;
            if (!hit) {
                tail = null_color;                        // :507-509
            } else if (is_light) {
                tail = scale(color, inten);               // :520-527
            } else if (rl.reflections_on && kref > 0.0f) {   // :595-604
                if (!dead) {
                    TCRT_CHECK(n_stacked >= 0 && n_stacked < CAP, kChkLevelStack);
                    float* rec = stack + 7 * n_stacked;
                    rec[0] = local.x; rec[1] = local.y; rec[2] = local.z;
                    rec[3] = kref;
                    rec[4] = color.x; rec[5] = color.y; rec[6] = color.z;
                    ++n_stacked;
                    // (k * child) * obj.c is +-0 for a finite child when obj.c == +-0: channel c of the pixel no longer
                    // depends on anything deeper.  rl.prune_dead: every child the reference forms is finite.
                    if (rl.prune_dead) {
                        ln.level |= ((color.x == 0.0f ? 1 : 0) | (color.y == 0.0f ? 2 : 0) | (color.z == 0.0f ? 4 : 0)) << kZeroShift;
                        if (ln.level >= kDead) ln.level |= n_stacked << kRecShift;
                    }
                }
                if ((ln.level & kLevelMask) + 1 > rl.max_depth) {
                    tail = null_color;                    // the child returns NULL_COLOR (:454-455)
                } else {
                    reflected = true;
                    ln.O = P;
                    ln.D = refl;
                    ++ln.level;
                    done = false;
                }
            } else {
                tail = local;
            }
            if (done) {
                if (dead) tail = mk(0.f, 0.f, 0.f);   // the deepest record's child: any finite colour gives the same pixel
                // final += (k * child) * obj, deepest level first (:601)
                TCRT_UNROLL_LOOP
                for (int i = n_stacked - 1; i >= 0; --i) {
                    TCRT_CHECK(i < CAP, kChkLevelStack);
                    const float* rec = stack + 7 * i;
#ifdef TCRT_CHECKED
                    for (int k = 0; k < 7; ++k) TCRT_CHECK(__float_as_uint(rec[k]) != 0x7fc0deadu, kChkPoison);
#endif
                    V3 kc = scale(tail, rec[3]);
                    tail.x = rec[0] + kc.x * rec[4];
                    tail.y = rec[1] + kc.y * rec[5];
                    tail.z = rec[2] + kc.z * rec[6];
                }
                TCRT_CHECK(ln.pix >= 0 && (unsigned)ln.pix < total, kChkPixel);
                float* o = rl.out + 3 * (size_t)ln.pix;
                o[0] = tail.x;
                o[1] = tail.y;
                o[2] = tail.z;
                // cost estimate for the band balancer's pre-pass: bounces of this pixel, per column
                if (MODE == kModeBand && rl.col_cost != nullptr) {
                    const int xc = ln.pix / rl.height;
                    const unsigned bounces = (unsigned)((ln.level & kLevelMask) + 1);
                    atomicAdd(rl.col_cost + xc, bounces);
                    atomicAdd(rl.col_cost + (rl.x1 - rl.x0) + (ln.pix - xc * rl.height), bounces);
                }
                ln.pix = -1;
            }
        }
        n_reflect += (unsigned)__popc(__ballot_sync(kFull, reflected));
    }

    // ---- ray counters: one atomic per warp and kind ---------------------------------------------
    if (lane == 0) {
        atomicAdd(rl.counters + 0, (unsigned long long)n_primary);
        atomicAdd(rl.counters + 1, (unsigned long long)n_shadow);
        atomicAdd(rl.counters + 2, (unsigned long long)n_reflect);
        if (MODE == kModeRays && n_invalid != 0) atomicAdd(rl.ray_invalid, (unsigned long long)n_invalid);
    }
}

template <int CAP, int FM>
__global__ void __launch_bounds__(kGridBlock, kGridMinBlocks) render_grid_kernel(const __grid_constant__ RenderLaunch rl) {
    render_grid_body<CAP, FM, kModeBand>(rl);
}

template <int CAP, int FM>
__global__ void __launch_bounds__(kGridBlock, kGridMinBlocks) render_grid_list_kernel(const __grid_constant__ RenderLaunch rl) {
    render_grid_body<CAP, FM, kModeList>(rl);
}

template <int CAP, int FM>
__global__ void __launch_bounds__(kGridBlock, kGridMinBlocks) render_grid_rays_kernel(const __grid_constant__ RenderLaunch rl) {
    render_grid_body<CAP, FM, kModeRays>(rl);
}

template <int CAP, int FM>
__global__ void __launch_bounds__(kGridBlock, kGridMinBlocks) render_grid_views_kernel(const __grid_constant__ RenderLaunch rl) {
    render_grid_body<CAP, FM, kModeViews>(rl);
}

template <int CAP, int FM>
cudaError_t launch_grid_one(const RenderLaunch& rl, int grid, size_t smem, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(render_grid_kernel<CAP, FM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    render_grid_kernel<CAP, FM><<<grid, kGridBlock, smem, stream>>>(rl);
    return cudaGetLastError();
}

// the list-, ray- and views-mode twins
template <int CAP, int FM>
cudaError_t launch_grid_list_one(const RenderLaunch& rl, int grid, size_t smem, cudaStream_t stream, RenderMode mode) {
    const auto kernel = mode == kModeViews ? render_grid_views_kernel<CAP, FM>
                        : mode == kModeRays ? render_grid_rays_kernel<CAP, FM>
                                            : render_grid_list_kernel<CAP, FM>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kernel<<<grid, kGridBlock, smem, stream>>>(rl);
    return cudaGetLastError();
}

template <int CAP>
cudaError_t launch_grid_cap(const RenderLaunch& rl, int fm, int grid, size_t smem, cudaStream_t stream, RenderMode mode) {
    if (mode != kModeBand)
        return fm == 0 ? launch_grid_list_one<CAP, 0>(rl, grid, smem, stream, mode) : launch_grid_list_one<CAP, 3>(rl, grid, smem, stream, mode);
    return fm == 0 ? launch_grid_one<CAP, 0>(rl, grid, smem, stream) : launch_grid_one<CAP, 3>(rl, grid, smem, stream);
}

}  // namespace

#ifdef TCRT_CHECKED
// the checked build's flags of this translation unit (tcrt_dev_check_flags reads those of tcrt_render.cu)
extern "C" int tcrt_dev_grid_check_flags(unsigned int* flags, int reset) {
    cudaDeviceSynchronize();
    if (flags && cudaMemcpyFromSymbol(flags, g_check_flags, sizeof(unsigned int)) != cudaSuccess) return -1;
    if (reset) {
        const unsigned int z = 0;
        if (cudaMemcpyToSymbol(g_check_flags, &z, sizeof z) != cudaSuccess) return -1;
    }
    return 0;
}
#endif

#ifdef TCRT_LANE_STATS
extern "C" int tcrt_dev_lane_stats_grid(unsigned long long* out16, int reset) {
    cudaDeviceSynchronize();
    if (out16 && cudaMemcpyFromSymbol(out16, g_lane_stats, sizeof(unsigned long long) * 16) != cudaSuccess) return -1;
    if (reset) {
        unsigned long long z[16] = {};
        if (cudaMemcpyToSymbol(g_lane_stats, z, sizeof z) != cudaSuccess) return -1;
    }
    return 0;
}
#endif

// fm: 0 no finite planes, 3 a handful swept linearly; rl.scene.grid_cells != nullptr (tcrt_upload_scene built a grid).
// mode kModeList / kModeRays / kModeViews: the list-, ray- or views-mode kernels (tcrt_launch_render_list / _rays /
// _views; rl.list_n = the launch's queue positions), with no more CTAs than there are claims.
cudaError_t tcrt_launch_render_grid(const RenderLaunch& rl, int fm, int sm_count, size_t smem, cudaStream_t stream, RenderMode mode) {
    int ctas_per_sm = kGridMinBlocks;
    while (ctas_per_sm > 1 && (smem + 1024) * ctas_per_sm > 220 * 1024) --ctas_per_sm;
    int grid = sm_count * ctas_per_sm;
    if (mode != kModeBand) grid = (int)std::min<long long>(grid, ((long long)rl.list_n + kGridBlock - 1) / kGridBlock);
    const int levels = rl.max_depth + 1;
    if (levels <= 8) return launch_grid_cap<8>(rl, fm, grid, smem, stream, mode);
    if (levels <= 16) return launch_grid_cap<16>(rl, fm, grid, smem, stream, mode);
    if (levels <= 64) return launch_grid_cap<64>(rl, fm, grid, smem, stream, mode);
    return launch_grid_cap<256>(rl, fm, grid, smem, stream, mode);
}
