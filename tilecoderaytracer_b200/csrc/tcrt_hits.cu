// tcrt_hits.cu — primary-hit buffers (tcrt_hit_buffers), picking (tcrt_pick), and the ray-batch queries that need no
// bounce loop: nearest hits (tcrt_intersect_rays) and occlusion (tcrt_occluded_rays, tcrt_occluded_lights).
//
// Per pixel, what the reference computes at level 0 of calculatePixel (RayTracer.cpp:448-638): the winner of
// getCollision (:50-89), that winner's distance, and the direction of the normal ray of its CollisionObject
// (SceneObject.h:47-105).  The ray, the sweep and the winner's normal are the render kernel's own code (tcrt_render.cu),
// so the buffers describe exactly the frame the render kernels draw.
//
// A kernel of its own rather than an output of the render kernels: their bounce loop has to fit the instruction cache
// (DESIGN.md §4.4), and a primary hit needs none of it — no light loop, no level stack, no refill.  One sweep per pixel.
// Scenes with a sphere grid walk the sphere BVH, which is always built alongside the grid and finds the same nearest hit
// (DESIGN.md §4.5); its per-ray fattening covers rays from any origin, so ray batches (tcrt_intersect_rays) walk it too.
#include "tcrt_render_common.cuh"

namespace {

// Stage the sweep blob, as render_kernel does (the BVH-covered spheres in front of stage_off stay global), and view it.
__device__ __forceinline__ Sm stage_blob(const DeviceScene& sc, float4* smem4, int stage_off) {
    const int n_stage = sc.blob_f4 - stage_off;
    for (int i = threadIdx.x; i < n_stage; i += kBlock) smem4[i] = __ldg(sc.blob + stage_off + i);
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
    return sm;
}

template <int SBVH, int FM>
__global__ void __launch_bounds__(kBlock, (SBVH && FM == 0) ? kMinBlocksBvh : kMinBlocks) hits_kernel(const __grid_constant__ HitLaunch hl) {
    extern __shared__ float4 smem4[];
    const RenderLaunch& rl = hl.rl;
    const DeviceScene& sc = rl.scene;
    const int stage_off = SBVH ? sc.stage_off : 0;
    const Sm sm = stage_blob(sc, smem4, stage_off);

    const unsigned lane = threadIdx.x & 31u;
    const bool rays = rl.ray_d != nullptr;
    const unsigned total = rays ? (unsigned)rl.list_n
                                : hl.xz != nullptr ? (unsigned)hl.n_list : (unsigned)(rl.x1 - rl.x0) * (unsigned)rl.height;
    unsigned n_invalid = 0;
    for (;;) {
        // one claim = 32 queue positions: one 4x8 tile of the band (BVH walks of a warp stay coherent), or 32 list entries
        // or rays
        unsigned q0 = 0;
        if (lane == 0) q0 = atomicAdd(rl.queue, 32u);
        q0 = __shfl_sync(kFull, q0, 0);
        if (q0 >= total) break;
        const unsigned q = q0 + lane;
        bool active = q < total;
        int xc = 0, z = 0;
        V3 O = mk(0.f, 0.f, 0.f), D = mk(1.f, 0.f, 0.f);
        if (active && rays) {
            // the caller's ray; an invalid one gets the markers and takes no part in the sweep
            if (!ray_from_batch(rl, (int)q, O, D)) {
                const float nan = __uint_as_float(0x7fc00000u);
                if (hl.object) hl.object[q] = -2;
                if (hl.distance) hl.distance[q] = nan;
                if (hl.normal) hl.normal[3 * (size_t)q] = hl.normal[3 * (size_t)q + 1] = hl.normal[3 * (size_t)q + 2] = nan;
                active = false;
                ++n_invalid;
            }
        } else if (active) {
            if (hl.xz != nullptr) {      // list mode: rl.x0 == 0, the pairs were range-checked by the host
                xc = __ldg(hl.xz + 2 * (size_t)q);
                z = __ldg(hl.xz + 2 * (size_t)q + 1);
            } else {
                queue_to_pixel(rl, (int)q, xc, z);
            }
            TCRT_CHECK(xc >= 0 && xc < rl.x1 - rl.x0 && z >= 0 && z < rl.height, kChkQueue);
            primary_ray(rl, xc, z, O, D);
        }
        float best;
        int bkey;
        sweep_nearest<SBVH, FM>(sm, sc, O, D, rl.far_dist, active, best, bkey);
        if (active) {
            int obj = -1;
            float dist = rl.far_dist;
            V3 n2 = mk(0.f, 0.f, 0.f);
            if (bkey >= 0) {
                // the winner block of render_kernel (tcrt_render.cu, "winner's hit record"), reduced to n2
                TCRT_CHECK(bkey < sc.n_sph + sc.n_fin + sc.n_inf, kChkPrimKey);
                obj = sm.idx[bkey];
                TCRT_CHECK(obj >= 0 && obj < rl.n_objects, kChkObject);
                dist = best;
                if (bkey < sc.n_sph) {
                    const V3 Pp = scale(D, best) + O;   // t*D + O  (SceneSphere.cpp:122)
                    const float4 sg = (SBVH && bkey < stage_off) ? __ldg(sc.blob + bkey) : sm.sph[bkey];
                    const V3 n1 = normalize(Pp - xyz(sg));   // SceneSphere.cpp:129-130
                    n2 = normalize(n1);                      // Ray(point, normal) re-normalises (Ray.h:21-25)
                } else {
                    float den;
                    if (bkey < sc.n_sph + sc.n_fin) {
                        TCRT_CHECK(bkey - sc.n_sph < sc.n_fin, kChkPrimKey);
                        den = dot(D, xyz(sm.fin[4 * (bkey - sc.n_sph)]));
                    } else {
                        den = dot(D, xyz(sm.inf[bkey - sc.n_sph - sc.n_fin]));
                    }
                    // computeNormal: normal.dot(eyeDir) < 0 ? normal : reverseNormal, re-normalised by Ray(point, normal):
                    // a constant of the plane side, tabulated at upload
                    n2 = xyz(__ldg(sc.obj_normals + 6 * obj + (den < 0.0f ? 0 : 3) + 1));
                }
            }
            const size_t pix = (rays || hl.xz != nullptr) ? (size_t)q : (size_t)xc * rl.height + z;
            TCRT_CHECK(pix < total, kChkPixel);
            if (hl.object) hl.object[pix] = obj;   // only ray batches may leave an output out
            if (hl.distance) hl.distance[pix] = dist;
            if (hl.normal) {
                hl.normal[3 * pix + 0] = n2.x;
                hl.normal[3 * pix + 1] = n2.y;
                hl.normal[3 * pix + 2] = n2.z;
            }
        }
    }
    if (rays) {
        const unsigned n = __reduce_add_sync(kFull, n_invalid);
        if (lane == 0 && n != 0) atomicAdd(rl.ray_invalid, (unsigned long long)n);
    }
}

// Occlusion queries (tcrt_occluded_rays / tcrt_occluded_lights): inShadeCollisionDetection (RayTracer.cpp:709-739) of a
// caller's ray with its own limit, or inShade (:743-771) of a caller's point against every light.  The any-hit walk is
// the render kernel's sweep_shadow; claims and staging are hits_kernel's.  A lane with nothing to ask (past the end, an
// invalid ray or pair) enters the warp-synchronous walks as a lane that wants no answer.
template <int SBVH, int FM>
__global__ void __launch_bounds__(kBlock, (SBVH && FM == 0) ? kMinBlocksBvh : kMinBlocks) occlusion_kernel(const __grid_constant__ OccLaunch ol) {
    extern __shared__ float4 smem4[];
    const RenderLaunch& rl = ol.rl;
    const DeviceScene& sc = rl.scene;
    const Sm sm = stage_blob(sc, smem4, SBVH ? sc.stage_off : 0);

    const unsigned lane = threadIdx.x & 31u;
    const bool points = ol.points != nullptr;
    const unsigned total = (unsigned)rl.list_n;
    unsigned n_invalid = 0, n_tests = 0;
    for (;;) {
        unsigned q0 = 0;
        if (lane == 0) q0 = atomicAdd(rl.queue, 32u);
        q0 = __shfl_sync(kFull, q0, 0);
        if (q0 >= total) break;
        const unsigned q = q0 + lane;
        const bool active = q < total;
        if (!points) {
            // the caller's ray and limit; no shell shortcut (mask 0): the far end of the segment is not a light
            V3 O = mk(0.f, 0.f, 0.f), D = mk(1.f, 0.f, 0.f);
            float tmax = 1.0f;
            bool want = false;
            if (active) {
                const float t = __ldg(ol.tmax + q);
                want = ray_from_batch(rl, (int)q, O, D) && t > 0.0f;   // NaN and t <= 0 fail
                if (want) tmax = t;
                else ol.out[q] = 0xFF;
            }
            const bool occl = sweep_shadow<SBVH, FM>(sm, sc, O, D, tmax, 0u, !want);
            if (want) ol.out[q] = occl ? 1 : 0;
            n_tests += want ? 1u : 0u;
            n_invalid += (active && !want) ? 1u : 0u;
        } else {
            // the point: the origin rule of ray batches
            V3 P = mk(0.f, 0.f, 0.f);
            bool ok = false;
            if (active) {
                const float* pp = ol.points + 3 * (size_t)q;
                P = mk(__ldg(pp), __ldg(pp + 1), __ldg(pp + 2));
                const float big = 1099511627776.0f;   // 2^40; NaN fails
                ok = fabsf(P.x) <= big && fabsf(P.y) <= big && fabsf(P.z) <= big;
                if (!ok) P = mk(0.f, 0.f, 0.f);
            }
            for (int l = 0; l < sc.n_lights; ++l) {   // warp-uniform: the light's shell mask is the warp's
                const float4 lp = sm.light[2 * l];
                const float4 lc = sm.light[2 * l + 1];
                // inShade (:743-752), as the render kernel's light loop builds it: dir = L - P, |dir|, Ray(P, dir)
                // normalises with the same length
                const V3 dir = xyz(lp) - P;
                const float dist = __fsqrt_rn(dir.x * dir.x + dir.y * dir.y + dir.z * dir.z);
                const V3 lr = div3(dir, dist);
                // the direction rule of ray batches; fails only within ~1e-19 of the light (0/0 at it)
                const float s = __fadd_rn(__fadd_rn(__fmul_rn(lr.x, lr.x), __fmul_rn(lr.y, lr.y)), __fmul_rn(lr.z, lr.z));
                const bool want = ok && fabsf(s - 1.0f) <= 4.76837158203125e-07f;
                const bool occl = sweep_shadow<SBVH, FM>(sm, sc, P, lr, dist, __float_as_uint(lc.w), !want);
                if (active) ol.out[(size_t)q * (unsigned)sc.n_lights + l] = want ? (occl ? 1 : 0) : 0xFF;
                n_tests += want ? 1u : 0u;
                n_invalid += (active && !want) ? 1u : 0u;
            }
        }
    }
    const unsigned t = __reduce_add_sync(kFull, n_tests);
    const unsigned n = __reduce_add_sync(kFull, n_invalid);
    if (lane == 0 && t != 0) atomicAdd(rl.counters + 1, (unsigned long long)t);
    if (lane == 0 && n != 0) atomicAdd(rl.ray_invalid, (unsigned long long)n);
}

template <int SBVH, int FM>
cudaError_t launch_occlusion_one(const OccLaunch& ol, int grid, size_t smem, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(occlusion_kernel<SBVH, FM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    occlusion_kernel<SBVH, FM><<<grid, kBlock, smem, stream>>>(ol);
    return cudaGetLastError();
}

template <int SBVH, int FM>
cudaError_t launch_hits_one(const HitLaunch& hl, int grid, size_t smem, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(hits_kernel<SBVH, FM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    hits_kernel<SBVH, FM><<<grid, kBlock, smem, stream>>>(hl);
    return cudaGetLastError();
}

}  // namespace

#ifdef TCRT_CHECKED
// the checked build's flags of this translation unit (tcrt_dev_check_flags reads those of tcrt_render.cu)
extern "C" int tcrt_dev_hits_check_flags(unsigned int* flags, int reset) {
    cudaDeviceSynchronize();
    if (flags && cudaMemcpyFromSymbol(flags, g_check_flags, sizeof(unsigned int)) != cudaSuccess) return -1;
    if (reset) {
        const unsigned int z = 0;
        if (cudaMemcpyToSymbol(g_check_flags, &z, sizeof z) != cudaSuccess) return -1;
    }
    return 0;
}
#endif

// The launch shape of the hit and occlusion kernels: staged bytes, a persistent grid sized as tcrt_launch_render sizes the
// render kernel's but with no more CTAs than `total` items need, and the dispatch class.  false: the blob does not fit.
static bool launch_shape(const RenderLaunch& rl, unsigned total, int sm_count, size_t& smem, int& grid, int& sb, int& fm) {
    smem = (size_t)std::max(1, rl.scene.blob_f4 - rl.scene.stage_off) * sizeof(float4);
    if (smem > tcrt_render_max_smem()) return false;
    int ctas_per_sm = (rl.scene.bvh_sph != nullptr && rl.scene.n_fin == 0) ? kMinBlocksBvh : kMinBlocks;
    while (ctas_per_sm > 1 && (smem + 1024) * ctas_per_sm > 220 * 1024) --ctas_per_sm;
    const long long need = ((long long)total + kBlock - 1) / kBlock;
    grid = (int)std::min<long long>((long long)sm_count * ctas_per_sm, need);
    sb = rl.scene.bvh_sph == nullptr ? 0 : 1;
    fm = rl.scene.bvh_fin != nullptr ? 2 : (rl.scene.n_fin == 0 ? 0 : (rl.scene.n_clu > 0 ? 1 : 3));
    return true;
}

cudaError_t tcrt_launch_hits(const HitLaunch& hl_in, int sm_count, cudaStream_t stream) {
    HitLaunch hl = hl_in;
    RenderLaunch& rl = hl.rl;
    const unsigned total = rl.ray_d != nullptr ? (unsigned)rl.list_n
                           : hl.xz != nullptr ? (unsigned)hl.n_list : (unsigned)(rl.x1 - rl.x0) * (unsigned)rl.height;
    size_t smem;
    int grid, sb, fm;
    if (!launch_shape(rl, total, sm_count, smem, grid, sb, fm)) return cudaErrorInvalidValue;
    if (total == 0) return cudaSuccess;
    rl.tiled = (hl.xz == nullptr && rl.ray_d == nullptr && (rl.x1 - rl.x0) % TCRT_TILE_W == 0 && rl.height % TCRT_TILE_H == 0) ? 1 : 0;
    rl.row_order = nullptr;
#define TCRT_CASE(SB, FMV) \
    if (sb == SB && fm == FMV) return launch_hits_one<SB, FMV>(hl, grid, smem, stream);
    TCRT_CASE(0, 0) TCRT_CASE(0, 1) TCRT_CASE(0, 2) TCRT_CASE(0, 3)
    TCRT_CASE(1, 0) TCRT_CASE(1, 1) TCRT_CASE(1, 2) TCRT_CASE(1, 3)
#undef TCRT_CASE
    return cudaErrorInvalidValue;
}

cudaError_t tcrt_launch_occlusion(const OccLaunch& ol_in, int sm_count, cudaStream_t stream) {
    OccLaunch ol = ol_in;
    const unsigned total = (unsigned)ol.rl.list_n;
    size_t smem;
    int grid, sb, fm;
    if (!launch_shape(ol.rl, total, sm_count, smem, grid, sb, fm)) return cudaErrorInvalidValue;
    if (total == 0) return cudaSuccess;
    ol.rl.tiled = 0;
    ol.rl.row_order = nullptr;
#define TCRT_CASE(SB, FMV) \
    if (sb == SB && fm == FMV) return launch_occlusion_one<SB, FMV>(ol, grid, smem, stream);
    TCRT_CASE(0, 0) TCRT_CASE(0, 1) TCRT_CASE(0, 2) TCRT_CASE(0, 3)
    TCRT_CASE(1, 0) TCRT_CASE(1, 1) TCRT_CASE(1, 2) TCRT_CASE(1, 3)
#undef TCRT_CASE
    return cudaErrorInvalidValue;
}
