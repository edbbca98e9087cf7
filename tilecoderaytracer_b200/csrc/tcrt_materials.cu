// tcrt_materials.cu — material edits (tcrt_update_materials, tcrt_update_textures): new colours, shading factors, light
// intensities, texture ids and checker rows for the resident scene, written in place by one scatter launch.
//
// No pruning structure depends on a material (DESIGN.md §4.5): the kernels read materials from these tables at run time,
// so rewriting the rows the upload would write is exact.  The host validates every record, merges it into its copy of the
// materials (for the dead-path bound) and sends full rows.  Of the scene, the launch reads only the light bit of each
// edited object's material row; it writes the rows the render, hit and occlusion launches read, never while one runs
// (the call waits for the render stream first).
#include "tcrt_device.h"

namespace {

constexpr int kMatBlock = 128;

__global__ void __launch_bounds__(kMatBlock) material_edit_kernel(const MaterialLaunch ml) {
    const int i = blockIdx.x * kMatBlock + threadIdx.x;
    if (i >= ml.n) return;
    const MaterialRecord r = ml.rec[i];
    if (r.target < 0) {   // a checker row: (light rgb, width) (dark rgb, height)
        const int t = ~r.target;
        ml.textures[2 * t] = r.a;
        ml.textures[2 * t + 1] = r.b;
        return;
    }
    const int o = r.target;
    // the w word as the upload packs it (plan_scene_blob): texture id + 1, and the light bit, which an edit keeps
    const unsigned light = __float_as_uint(ml.material[o].w) & 0x80000000u;
    float4 m = r.b;
    m.w = __uint_as_float(((unsigned)(r.tex + 1) & 0x7fffffffu) | light);
    ml.surface[o] = r.a;
    ml.material[o] = m;
    const int l = ml.light_of[o];
    if (l >= 0) {   // the light table (light_rows, tcrt_api.cu): the position and the inside mask stay where they are
        float4* row = ml.lights + 2 * l;
        row[0].w = r.b.z;
        row[1].x = r.a.x;
        row[1].y = r.a.y;
        row[1].z = r.a.z;
    }
}

}  // namespace

cudaError_t tcrt_launch_material_edit(const MaterialLaunch& ml, cudaStream_t stream, int* launches) {
    if (ml.n <= 0) return cudaSuccess;
    material_edit_kernel<<<(ml.n + kMatBlock - 1) / kMatBlock, kMatBlock, 0, stream>>>(ml);
    *launches += 1;
    return cudaGetLastError();
}
