// tcrt_render.cu — the per-pixel render path as a persistent sm_100a kernel.
//
// Replaces, in the reference: the pixel loop (RayTracer.cpp:911-923), Camera::createEyeRay
// (Camera.cpp:71-84), calculatePixel (RayTracer.cpp:448-638), getCollision (:50-89), the three
// SceneObject::collision overrides (SceneSphere.cpp:50-168, SceneFinitePlane.cpp:86-164,
// SceneInfinitePlane.cpp:29-108), the CollisionObject ctor (SceneObject.h:47-105), cosineShade
// (:654-701), inShade/inShadeCollisionDetection (:709-771), Texture_CheckerBoard lookup
// (Texture_CheckerBoard.h:31-65) and — as work distribution — PixelQueue / the TILE64
// strategies (PixelQueue.cpp, RayTracer.cpp:956-1079).
//
// Shape (B200-first, not a translation):
//   * per-type SoA primitive arrays staged once per CTA into shared memory with coalesced
//     float4 loads; every lane of a warp walks the same primitive (shared-memory broadcast),
//     so there is no virtual dispatch and no divergence on the primitive type;
//   * pruning that cannot change a result (DESIGN.md §4.5): a division-free prefilter in front
//     of every plane test, box clusters for axis-aligned rectangles (every makeSceneBox face),
//     a BVH per type for scenes with many primitives.  Whatever survives is evaluated with the
//     reference's exact operation sequence, ties resolved on the object index;
//   * recursion -> an iterative "bounce" loop.  A lane's ray state lives in registers; the
//     only per-level storage is (local colour, k, object colour) in a small local-memory
//     stack, folded from the deepest level up so that  final += k*child*obj
//     (RayTracer.cpp:601) keeps the reference's association bit for bit;
//   * persistent warps + an atomic pixel queue: a warp claims 32 queue positions (a 4x8-pixel
//     tile) with one atomicAdd and, before every bounce, ballots for lanes whose
//     path has ended; once enough of them are idle (rl.refill_min) exactly those lanes get fresh
//     primary rays.  Reflection tails (65% / 13% / ... of pixels alive per level, SURVEY §6.2)
//     therefore do not leave lanes idle: a bounce is the same code for a primary ray and a
//     depth-40 mirror ray;
//   * the bounce loop has to fit the 32 KB instruction cache: rare code is out of line, sweep
//     loops are not unrolled, scene-dependent code is selected by template parameters;
//   * arithmetic is IEEE binary32 with no contraction (nvcc -fmad=false), '/' and sqrtf
//     correctly rounded (__fdiv_rn / __fsqrt_rn, or the same instruction sequence with a shared
//     reciprocal, div3), matching vector3d.h with USING_FIXED_POINT false.  The expression order
//     of every formula is the reference's; FFMA appears only inside division / square-root
//     sequences and in pruning tests.
#include "tcrt_render_common.cuh"

namespace {

// The kernel body.  MODE kModeBand: the pixels of the band [rl.x0, rl.x1) (render_kernel).  kModeList: the samples of a
// pixel list (render_list_kernel, adaptive frames; RenderLaunch::list).  kModeRays: the caller's rays (render_rays_kernel,
// ray batches; RenderLaunch::ray_*).  kModeViews: band mode over the global columns of a stack of views whose primary rays
// take their camera from a table (render_views_kernel, multi-view frames; RenderLaunch::view_cams).  Only the refill
// block, the output slot and the invalid-ray count differ.
template <int CAP, int SBVH, int FM, int MODE>
__device__ __forceinline__ void render_body(const RenderLaunch& rl) {
    extern __shared__ float4 smem4[];
    const DeviceScene& sc = rl.scene;
    // ---- stage the sweep blob: coalesced 16-byte loads, once per CTA ------------------------
    // (the BVH-covered spheres in front of stage_off stay in global memory)
    const int stage_off = SBVH ? sc.stage_off : 0;   // compile-time 0 without a sphere BVH
    const int n_stage = sc.blob_f4 - stage_off;
    for (int i = threadIdx.x; i < n_stage; i += kBlock) smem4[i] = __ldg(sc.blob + stage_off + i);
    __syncthreads();
    Sm sm;
    const float4* base = smem4 - stage_off;     // blob offsets -> shared memory
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
    for (int i = 0; i < CAP * 7; ++i) stack[i] = __uint_as_float(0x7fc0dead);   // poison: a quiet NaN nothing computes
#endif
    Lane ln;
    ln.pix = -1;
    ln.level = 0;
    ln.O = mk(0.f, 0.f, 0.f);
    ln.D = mk(1.f, 0.f, 0.f);
    // ray counters: per WARP (ballot + popc keeps them in uniform registers, not in every lane's)
    unsigned n_primary = 0, n_shadow = 0, n_reflect = 0;
    unsigned n_invalid = 0;        // ray mode: rays refused by the validity rule
    unsigned wcur = 0, wend = 0;   // the warp's claimed chunk of pixel ids
    bool exhausted = false;

    for (;;) {
        // ---- refill: lanes whose path ended take the next pixel ids of the warp's chunk ------
        unsigned idle = __ballot_sync(kFull, ln.pix < 0);
        while (__popc(idle) >= rl.refill_min && !exhausted) {
            if (wcur == wend) {
                // one claim = 32 queue positions (one pixel per lane, one 4x8 tile).  Larger or guided
                // claims were measured: a claim cannot be split once taken, and where deep reflection
                // paths are concentrated (the mirror tunnel of SCENE 2, the default scene at depth 50) a
                // warp holding several tiles of them becomes the tail of the launch.
                unsigned base = 0;
                if (lane == 0) base = atomicAdd(rl.queue, 32u);
                base = __shfl_sync(kFull, base, 0);
                if (base >= total) {
                    exhausted = true;
                    break;
                }
                wcur = base;
                wend = min(base + 32u, total);
            }
            unsigned avail = wend - wcur;
            unsigned rank = __popc(idle & lt_mask);
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
                    TCRT_CHECK(xc >= 0 && xc < rl.x1 - rl.x0 && z >= 0 && z < rl.height, kChkQueue);
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
        TCRT_STAT(0, ~idle);

        // ---- nearest hit -----------------------------------------------------------------
        float best;
        int bkey;
        sweep_nearest<SBVH, FM>(sm, sc, ln.O, ln.D, rl.far_dist, active, best, bkey);
        const bool hit = active && bkey >= 0;

        // ---- winner's hit record (CollisionObject ctor, SceneObject.h:47-105) -------------------
        V3 P = ln.O, n2 = mk(0.f, 0.f, 1.f), N = n2, refl = ln.D, color = null_color;
        float diffuse = 0.f, specular = 0.f, kref = 0.f, inten = 0.f;
        bool is_light = false;
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
            const int tex = (flags & 0x7fffffff) - 1;
            V3 n1;
            V3 Pp = scale(ln.D, best) + ln.O;   // t*D + O  (SceneSphere.cpp:122, SceneFinitePlane.cpp:108)
            if (bkey < sc.n_sph) {
                P = Pp;
                const float4 sg = (SBVH && bkey < stage_off) ? __ldg(sc.blob + bkey) : sm.sph[bkey];
                n1 = normalize(Pp - xyz(sg));   // SceneSphere.cpp:129-130
                n2 = normalize(n1);                       // Ray(point, normal) re-normalises (Ray.h:21-25)
                N = normalize(n2);                        // specular's N: normalised once more (:565-566)
            } else {
                float den;
                float px = 0.f, py = 0.f;
                if (bkey < sc.n_sph + sc.n_fin) {
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
                // computeNormal: normal.dot(eyeDir) < 0 ? normal : reverseNormal; its two
                // re-normalisations (Ray(point, normal), Ray.h:21-25; specular N, RayTracer.cpp:565-566)
                // are constants of the plane side, tabulated at upload
                const float4* nt = sc.obj_normals + 6 * obj + (den < 0.0f ? 0 : 3);
                n1 = xyz(__ldg(nt));
                n2 = xyz(__ldg(nt + 1));
                N = xyz(__ldg(nt + 2));
                // + temp_normal * INTERSECTION_OFFSET_DIST (1E-3 narrowed to float)
                P = Pp + scale(n1, 0.0010000000475f);
            }
            if (kref > 0.0f && !is_light) {
                float ndi = dot(n1, ln.D);     // SceneObject.h:63
                // -2*normal.k * n_dot_incoming + incoming.k  (SceneObject.h:81-83), then Ray() normalises
                refl = normalize(mk(-2.0f * n1.x * ndi + ln.D.x, -2.0f * n1.y * ndi + ln.D.y,
                                    -2.0f * n1.z * ndi + ln.D.z));
            }
        }

        // ---- light loop (RayTracer.cpp:537-591) ----------------------------------------------
        const bool shade = hit && !is_light;
        V3 local = mk(0.f, 0.f, 0.f);
        if (__any_sync(kFull, shade)) {
            TCRT_STAT(12, __ballot_sync(kFull, shade));
            for (int l = 0; l < sc.n_lights; ++l) {
                const float4 lp = sm.light[2 * l];
                const float4 lc = sm.light[2 * l + 1];
                // inShade (:743-752): dir = L - P, |dir|, Ray(P, dir) normalises with the same length
                V3 dir = xyz(lp) - P;
                float dist = __fsqrt_rn(dir.x * dir.x + dir.y * dir.y + dir.z * dir.z);
                V3 lr = div3(dir, dist);
                bool occl = !shade;
                if (rl.shadows_on) {
                    n_shadow += (unsigned)__popc(__ballot_sync(kFull, shade));
                    // The answer only matters if this light can change `local`: a positive cosine term,
                    // the clamp of cosineShade (which runs for every unshadowed light once local > 1), or
                    // a positive specular dot product.  Otherwise the ray is counted but not traced.
                    // (Only where a shadow ray is a BVH walk: for the linear sweeps of a small scene the two
                    // extra dot products cost more than the skipped sweeps return — measured.)
                    bool matters = true;
                    if (SBVH) {
                        const float c_pre = dot(n2, lr);
                        const float d_pre = dot(ln.D, lr - scale(N, 2.0f * dot(lr, N)));
                        matters = (d_pre > 0.0f) || (diffuse > 0.0f && (c_pre > 0.0f || local.x > 1.0f || local.y > 1.0f ||
                                                                         local.z > 1.0f));
                    }
                    TCRT_STAT(10, __ballot_sync(kFull, !(occl || !matters)));
                    occl = sweep_shadow<SBVH, FM>(sm, sc, P, lr, dist, __float_as_uint(lc.w), occl || !matters);
                }
                if (!occl) {
                    // cosineShade (:654-701); its light_ray equals lr
                    if (diffuse > 0.0f) {
                        float c = dot(n2, lr);
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
                    float two_ln = 2.0f * dot(lr, N);
                    V3 R = lr - scale(N, two_ln);
                    float d = dot(ln.D, R);
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
        }

        // ---- continue or finish the path --------------------------------------------------------
        bool reflected = false;
        if (active) {
            V3 tail;
            bool done = true;
            int n_stacked = ln.level;
            if (!hit) {
                tail = null_color;                        // :507-509
            } else if (is_light) {
                tail = scale(color, inten);               // :520-527
            } else if (rl.reflections_on && kref > 0.0f) {   // :595-604
                TCRT_CHECK(ln.level >= 0 && ln.level < CAP, kChkLevelStack);
                float* rec = stack + 7 * ln.level;   // every level below this one stacked a record
                rec[0] = local.x; rec[1] = local.y; rec[2] = local.z;
                rec[3] = kref;
                rec[4] = color.x; rec[5] = color.y; rec[6] = color.z;
                ++n_stacked;
                if (ln.level + 1 > rl.max_depth) {
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
                    atomicAdd(rl.col_cost + xc, (unsigned)(ln.level + 1));
                    atomicAdd(rl.col_cost + (rl.x1 - rl.x0) + (ln.pix - xc * rl.height), (unsigned)(ln.level + 1));
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

template <int CAP, int SBVH, int FM>
__global__ void __launch_bounds__(kBlock, (SBVH && FM == 0) ? kMinBlocksBvh : kMinBlocks) render_kernel(const __grid_constant__ RenderLaunch rl) {
    render_body<CAP, SBVH, FM, kModeBand>(rl);
}

template <int CAP, int SBVH, int FM>
__global__ void __launch_bounds__(kBlock, (SBVH && FM == 0) ? kMinBlocksBvh : kMinBlocks) render_list_kernel(const __grid_constant__ RenderLaunch rl) {
    render_body<CAP, SBVH, FM, kModeList>(rl);
}

template <int CAP, int SBVH, int FM>
__global__ void __launch_bounds__(kBlock, (SBVH && FM == 0) ? kMinBlocksBvh : kMinBlocks) render_rays_kernel(const __grid_constant__ RenderLaunch rl) {
    render_body<CAP, SBVH, FM, kModeRays>(rl);
}

template <int CAP, int SBVH, int FM>
__global__ void __launch_bounds__(kBlock, (SBVH && FM == 0) ? kMinBlocksBvh : kMinBlocks) render_views_kernel(const __grid_constant__ RenderLaunch rl) {
    render_body<CAP, SBVH, FM, kModeViews>(rl);
}

template <int CAP, int SBVH, int FM>
cudaError_t launch_one(const RenderLaunch& rl, int grid, size_t smem, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(render_kernel<CAP, SBVH, FM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return e;
    render_kernel<CAP, SBVH, FM><<<grid, kBlock, smem, stream>>>(rl);
    return cudaGetLastError();
}

template <int CAP>
cudaError_t launch_cap(const RenderLaunch& rl, int grid, size_t smem, cudaStream_t stream) {
    const int sb = rl.scene.bvh_sph == nullptr ? 0 : 1;
    const int fm = rl.scene.bvh_fin != nullptr ? 2 : (rl.scene.n_fin == 0 ? 0 : (rl.scene.n_clu > 0 ? 1 : 3));
#define TCRT_CASE(SB, FMV) \
    if (sb == SB && fm == FMV) return launch_one<CAP, SB, FMV>(rl, grid, smem, stream);
    TCRT_CASE(0, 0) TCRT_CASE(0, 1) TCRT_CASE(0, 2) TCRT_CASE(0, 3)
    TCRT_CASE(1, 0) TCRT_CASE(1, 1) TCRT_CASE(1, 2) TCRT_CASE(1, 3)
#undef TCRT_CASE
    return cudaErrorInvalidValue;
}

// the list-, ray- and views-mode twins (kModeList, kModeRays, kModeViews)
template <int CAP, int SBVH, int FM, int MODE>
cudaError_t launch_list_one(const RenderLaunch& rl, int grid, size_t smem, cudaStream_t stream) {
    const auto kernel = MODE == kModeViews ? render_views_kernel<CAP, SBVH, FM>
                        : MODE == kModeRays ? render_rays_kernel<CAP, SBVH, FM>
                                            : render_list_kernel<CAP, SBVH, FM>;
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    kernel<<<grid, kBlock, smem, stream>>>(rl);
    return cudaGetLastError();
}

template <int CAP, int MODE>
cudaError_t launch_list_cap(const RenderLaunch& rl, int grid, size_t smem, cudaStream_t stream) {
    const int sb = rl.scene.bvh_sph == nullptr ? 0 : 1;
    const int fm = rl.scene.bvh_fin != nullptr ? 2 : (rl.scene.n_fin == 0 ? 0 : (rl.scene.n_clu > 0 ? 1 : 3));
#define TCRT_CASE(SB, FMV) \
    if (sb == SB && fm == FMV) return launch_list_one<CAP, SB, FMV, MODE>(rl, grid, smem, stream);
    TCRT_CASE(0, 0) TCRT_CASE(0, 1) TCRT_CASE(0, 2) TCRT_CASE(0, 3)
    TCRT_CASE(1, 0) TCRT_CASE(1, 1) TCRT_CASE(1, 2) TCRT_CASE(1, 3)
#undef TCRT_CASE
    return cudaErrorInvalidValue;
}

}  // namespace

// ---- self-test of div3 against __fdiv_rn (tcrt_selftest_div3) ------------------------------------------
namespace {
__device__ __forceinline__ unsigned mix32(unsigned x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
__global__ void div3_check_kernel(unsigned long long n, unsigned seed, unsigned long long* bad) {
    unsigned long long local_bad = 0;
    for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned h0 = mix32((unsigned)i ^ seed), h1 = mix32(h0 + 0x9e3779b9u + (unsigned)(i >> 32));
        const unsigned h2 = mix32(h1 ^ 0x85ebca6bu), h3 = mix32(h2 + 0xc2b2ae35u), h4 = mix32(h3 ^ seed);
        // divisor: positive, exponent 2^-50 .. 2^50 (both sides of the fast-path window), any mantissa
        const unsigned eb = 77u + h0 % 101u;
        const float b = __uint_as_float((eb << 23) | (h1 & 0x7fffffu));
        float a[3];
        const unsigned hs[3] = {h2, h3, h4};
        for (int k = 0; k < 3; k++) {
            const unsigned h = hs[k], mode = h >> 29;
            float v;
            if (mode < 4u) {          // |a| <= b, uniform mantissa/scale
                v = b * ((float)(h & 0xffffffu) * (1.0f / 16777216.0f)) * ((h >> 24) & 1u ? -1.0f : 1.0f);
            } else if (mode < 6u) {   // any smaller exponent (down to denormals and zero), any mantissa
                const unsigned ea = (h >> 8) % (eb + 1u);
                v = __uint_as_float(((h >> 28) & 1u) << 31 | (ea << 23) | (mix32(h) & 0x7fffffu));
                if (fabsf(v) > b) v = b;
            } else if (mode == 6u) {
                v = (h & 1u) ? b : -b;
            } else {
                v = (h & 1u) ? 0.0f : -0.0f;
            }
            a[k] = v;
        }
        const V3 q = div3(mk(a[0], a[1], a[2]), b);
        const float r0 = __fdiv_rn(a[0], b), r1 = __fdiv_rn(a[1], b), r2 = __fdiv_rn(a[2], b);
        if (__float_as_uint(q.x) != __float_as_uint(r0) || __float_as_uint(q.y) != __float_as_uint(r1) ||
            __float_as_uint(q.z) != __float_as_uint(r2))
            ++local_bad;
    }
    if (local_bad) atomicAdd(bad, local_bad);
}
}  // namespace

cudaError_t tcrt_launch_div3_check(unsigned long long n, unsigned seed, unsigned long long* bad, cudaStream_t stream) {
    div3_check_kernel<<<148 * 8, 256, 0, stream>>>(n, seed, bad);
    return cudaGetLastError();
}

#ifdef TCRT_LANE_STATS
extern "C" int tcrt_dev_lane_stats(unsigned long long* out16, int reset) {
    cudaDeviceSynchronize();
    if (out16 && cudaMemcpyFromSymbol(out16, g_lane_stats, sizeof(unsigned long long) * 16) != cudaSuccess) return -1;
    if (reset) {
        unsigned long long z[16] = {};
        if (cudaMemcpyToSymbol(g_lane_stats, z, sizeof z) != cudaSuccess) return -1;
    }
    return 0;
}
#endif

#ifdef TCRT_CHECKED
extern "C" int tcrt_dev_check_flags(unsigned int* flags, int reset) {
    cudaDeviceSynchronize();
    if (flags && cudaMemcpyFromSymbol(flags, g_check_flags, sizeof(unsigned int)) != cudaSuccess) return -1;
    if (reset) {
        const unsigned int z = 0;
        if (cudaMemcpyToSymbol(g_check_flags, &z, sizeof z) != cudaSuccess) return -1;
    }
    return 0;
}
#endif

size_t tcrt_render_max_smem() { return 200 * 1024; }

static int finite_mode(const DeviceScene& sc) {
    return sc.bvh_fin != nullptr ? 2 : (sc.n_fin == 0 ? 0 : (sc.n_clu > 0 ? 1 : 3));
}

size_t tcrt_wave_mem_needed(const RenderLaunch& rl) {
#ifdef TCRT_DEV_KNOBS   // the experimental wavefront path (tcrt_render_wave.cu) exists in developer builds only
    if (getenv("TCRT_WAVE") == nullptr || !tcrt_wave_applies(rl, finite_mode(rl.scene))) return 0;
    return tcrt_wave_mem_bytes((size_t)(rl.x1 - rl.x0) * rl.height, rl.max_depth);
#else
    (void)rl;
    return 0;
#endif
}

cudaError_t tcrt_launch_render(const RenderLaunch& rl_in, int sm_count, cudaStream_t stream, int* launches, void* wave_mem,
                               size_t wave_bytes) {
    RenderLaunch rl = rl_in;
    const size_t smem_scene = (size_t)std::max(1, rl.scene.blob_f4 - rl.scene.stage_off) * sizeof(float4);
    if (smem_scene > tcrt_render_max_smem()) return cudaErrorInvalidValue;
    const int fm = finite_mode(rl.scene);
    const size_t smem = smem_scene;
#ifdef TCRT_DEV_KNOBS   // A/B: the experimental wavefront path (TCRT_WAVE=1), large frames of sphere-BVH scenes
    {
        const size_t need = tcrt_wave_mem_needed(rl);
        if (need != 0 && wave_mem != nullptr && wave_bytes >= need)
            return tcrt_launch_render_wave(rl, fm, sm_count, smem_scene, wave_mem, wave_bytes, stream, launches);
    }
#else
    (void)wave_mem;
    (void)wave_bytes;
#endif
    // persistent grid: kMinBlocks CTAs per SM (the register budget __launch_bounds__ asked for),
    // fewer when the staged scene does not fit that many times into shared memory
    int ctas_per_sm = (rl.scene.bvh_sph != nullptr && rl.scene.n_fin == 0) ? kMinBlocksBvh : kMinBlocks;
    while (ctas_per_sm > 1 && (smem + 1024) * ctas_per_sm > 220 * 1024) --ctas_per_sm;
    const int grid = sm_count * ctas_per_sm;
    rl.tiled = ((rl.x1 - rl.x0) % TCRT_TILE_W == 0 && rl.height % TCRT_TILE_H == 0) ? 1 : 0;
    // A warp takes new pixels once this many of its lanes are idle.  With one 4x8 tile per claim the
    // best value is 32 on every scene measured (profiles/README.md): the warp finishes its tile, then
    // takes the next.  Refilling part of a warp pays the primary-ray code more often and mixes tiles
    // and depths in one warp; before tiles (column strips, large claims) 12-20 was better.
    rl.refill_min = 32;
#ifdef TCRT_DEV_KNOBS   // developer build only (A/B timing); the product never reads the environment
    if (const char* e = getenv("TCRT_REFILL_MIN")) {
        const int v = atoi(e);
        if (v >= 1 && v <= 32) rl.refill_min = v;
    }
#endif
    cudaError_t e;
    const int levels = rl.max_depth + 1;   // levels 0..max_depth can each stack one record
    // spheres in a uniform grid (tcrt_upload_scene builds one only without finite-plane structures): tcrt_render_grid.cu
    if (rl.scene.grid_cells != nullptr && rl.scene.bvh_sph != nullptr && (fm == 0 || fm == 3)) {
        bool use_grid = true;
#ifdef TCRT_DEV_KNOBS
        if (getenv("TCRT_NO_GRID")) use_grid = false;
#endif
        if (use_grid) {
            e = tcrt_launch_render_grid(rl, fm, sm_count, smem, stream);
            if (launches) *launches += 1;
            return e;
        }
    }
    bool pool = false;
#ifdef TCRT_DEV_KNOBS   // the warp task pool (tcrt_render_pool.cu), for A/B timing against the kernels here
    pool = rl.scene.bvh_sph != nullptr && (fm == 0 || fm == 3) && getenv("TCRT_POOL") != nullptr;
#endif
    if (pool) {
        e = tcrt_launch_render_pool(rl, fm, sm_count, smem_scene, stream);
        if (launches) *launches += 1;
        return e;
    }
    if (levels <= 8) e = launch_cap<8>(rl, grid, smem, stream);
    else if (levels <= 16) e = launch_cap<16>(rl, grid, smem, stream);
    else if (levels <= 64) e = launch_cap<64>(rl, grid, smem, stream);
    else e = launch_cap<256>(rl, grid, smem, stream);
    if (launches) *launches += 1;
    return e;
}

// List mode (adaptive frames), ray mode (ray batches) and views mode (multi-view frames): the same kernels with the list,
// ray or views refill, grid-sized and dispatched as tcrt_launch_render does, never the developer builds' pool or wavefront
// paths.  One launch; nothing when the list is empty.  Views launches keep the band's 4x8 tiles (eye rays in x-major
// order trace 8-16 % slower than in tile order, profiles/README.md 12); the list is their band's pixels.
template <int MODE>
static cudaError_t launch_twin(const RenderLaunch& rl_in, int sm_count, cudaStream_t stream) {
    RenderLaunch rl = rl_in;
    if (MODE == kModeViews) rl.list_n = rl.x1 > rl.x0 ? (rl.x1 - rl.x0) * rl.height : 0;
    if (rl.list_n <= 0) return cudaSuccess;
    const size_t smem = (size_t)std::max(1, rl.scene.blob_f4 - rl.scene.stage_off) * sizeof(float4);
    if (smem > tcrt_render_max_smem()) return cudaErrorInvalidValue;
    const int fm = finite_mode(rl.scene);
    rl.tiled = MODE == kModeViews && (rl.x1 - rl.x0) % TCRT_TILE_W == 0 && rl.height % TCRT_TILE_H == 0 ? 1 : 0;
    rl.row_order = nullptr;
    rl.col_cost = nullptr;
    rl.refill_min = 32;
    if (rl.scene.grid_cells != nullptr && rl.scene.bvh_sph != nullptr && (fm == 0 || fm == 3))
        return tcrt_launch_render_grid(rl, fm, sm_count, smem, stream, (RenderMode)MODE);
    int ctas_per_sm = (rl.scene.bvh_sph != nullptr && rl.scene.n_fin == 0) ? kMinBlocksBvh : kMinBlocks;
    while (ctas_per_sm > 1 && (smem + 1024) * ctas_per_sm > 220 * 1024) --ctas_per_sm;
    // persistent grid, but no more CTAs than there are claims of 32 queue positions per warp
    const long long need = ((long long)rl.list_n + kBlock - 1) / kBlock;
    const int grid = (int)std::min<long long>((long long)sm_count * ctas_per_sm, need);
    const int levels = rl.max_depth + 1;
    if (levels <= 8) return launch_list_cap<8, MODE>(rl, grid, smem, stream);
    if (levels <= 16) return launch_list_cap<16, MODE>(rl, grid, smem, stream);
    if (levels <= 64) return launch_list_cap<64, MODE>(rl, grid, smem, stream);
    return launch_list_cap<256, MODE>(rl, grid, smem, stream);
}

cudaError_t tcrt_launch_render_list(const RenderLaunch& rl, int sm_count, cudaStream_t stream) {
    return launch_twin<kModeList>(rl, sm_count, stream);
}

cudaError_t tcrt_launch_render_rays(const RenderLaunch& rl, int sm_count, cudaStream_t stream) {
    return launch_twin<kModeRays>(rl, sm_count, stream);
}

cudaError_t tcrt_launch_render_views(const RenderLaunch& rl, int sm_count, cudaStream_t stream) {
    return launch_twin<kModeViews>(rl, sm_count, stream);
}
