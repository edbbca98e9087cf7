// tcrt_hits.cu — primary-hit buffers (tcrt_hit_buffers) and picking (tcrt_pick).
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

template <int SBVH, int FM>
__global__ void __launch_bounds__(kBlock, (SBVH && FM == 0) ? kMinBlocksBvh : kMinBlocks) hits_kernel(const __grid_constant__ HitLaunch hl) {
    extern __shared__ float4 smem4[];
    const RenderLaunch& rl = hl.rl;
    const DeviceScene& sc = rl.scene;
    // ---- stage the sweep blob, as render_kernel does (the BVH-covered spheres in front of stage_off stay global) ----
    const int stage_off = SBVH ? sc.stage_off : 0;
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

cudaError_t tcrt_launch_hits(const HitLaunch& hl_in, int sm_count, cudaStream_t stream) {
    HitLaunch hl = hl_in;
    RenderLaunch& rl = hl.rl;
    const size_t smem = (size_t)std::max(1, rl.scene.blob_f4 - rl.scene.stage_off) * sizeof(float4);
    if (smem > tcrt_render_max_smem()) return cudaErrorInvalidValue;
    const unsigned total = rl.ray_d != nullptr ? (unsigned)rl.list_n
                           : hl.xz != nullptr ? (unsigned)hl.n_list : (unsigned)(rl.x1 - rl.x0) * (unsigned)rl.height;
    if (total == 0) return cudaSuccess;
    // persistent grid, sized as tcrt_launch_render sizes the render kernel's, but no more CTAs than there are claims
    int ctas_per_sm = (rl.scene.bvh_sph != nullptr && rl.scene.n_fin == 0) ? kMinBlocksBvh : kMinBlocks;
    while (ctas_per_sm > 1 && (smem + 1024) * ctas_per_sm > 220 * 1024) --ctas_per_sm;
    const long long need = ((long long)total + kBlock - 1) / kBlock;
    const int grid = (int)std::min<long long>((long long)sm_count * ctas_per_sm, need);
    rl.tiled = (hl.xz == nullptr && rl.ray_d == nullptr && (rl.x1 - rl.x0) % TCRT_TILE_W == 0 && rl.height % TCRT_TILE_H == 0) ? 1 : 0;
    rl.row_order = nullptr;
    const int sb = rl.scene.bvh_sph == nullptr ? 0 : 1;
    const int fm = rl.scene.bvh_fin != nullptr ? 2 : (rl.scene.n_fin == 0 ? 0 : (rl.scene.n_clu > 0 ? 1 : 3));
#define TCRT_CASE(SB, FMV) \
    if (sb == SB && fm == FMV) return launch_hits_one<SB, FMV>(hl, grid, smem, stream);
    TCRT_CASE(0, 0) TCRT_CASE(0, 1) TCRT_CASE(0, 2) TCRT_CASE(0, 3)
    TCRT_CASE(1, 0) TCRT_CASE(1, 1) TCRT_CASE(1, 2) TCRT_CASE(1, 3)
#undef TCRT_CASE
    return cudaErrorInvalidValue;
}
