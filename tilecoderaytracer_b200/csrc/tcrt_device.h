// tcrt_device.h — internal: structures shared by the CUDA kernels and the C-ABI layer.
#ifndef TCRT_DEVICE_H_
#define TCRT_DEVICE_H_

#include <cuda_runtime.h>
#include <stdint.h>

#include "tcrt.h"

// ---- device-resident scene ---------------------------------------------------------------
// One allocation per device.  The "sweep blob" is what every CTA stages into shared memory
// with coalesced float4 loads; everything else is winner-only data read through the
// read-only path.
//
// Sweep blob layout (float4 units):
//   [0, n_sph)                      sphere   (cx, cy, cz, r^2)
//   [fin_off, fin_off + 4*n_fin)    finite   (n, -dto) (h, h_dist) (v, v_dist) (plane_origin, 0)
//   [inf_off, inf_off + n_inf)      infinite (n, -dto)
//   [light_off, light_off + 2*n_lights)  (light position, intensity) (light colour, 0)
//   [clu_off, clu_off + 4*n_clu)    box clusters of axis-aligned finite planes (tcrt_cluster.cpp):
//                                   (lo.x, hi.x, lo.y, hi.y) (lo.z, hi.z, present mask, -) (c of faces x0 x1 y0 y1) (c of z0 z1, -, -)
//                                   (pairs: one packed FADD2/FMUL2 handles both bounds / both faces of an axis)
//   [cslot_off, ...)                int32 finite-plane slot per cluster face (6 per cluster, -1 = absent)
//   [idx_off, ...)                  int32 object index per primitive: spheres, finite, infinite
// Within each type the non-light primitives come first (counts *_nl): the shadow sweep
// (inShadeCollisionDetection skips lights, RayTracer.cpp:727) just stops there.  The
// nearest-hit order inside a type is irrelevant because ties are resolved on the object
// index explicitly.
struct DeviceScene {
    const float4* blob;        // sweep blob (global)
    int blob_f4;               // size in float4 units (including the index tail, rounded up)
    int stage_off;             // CTAs stage blob[stage_off, blob_f4) into shared memory: the spheres a BVH covers
                               // (the first n_sph_bvh) are read from global memory through L1
    int n_sph, n_fin, n_inf;
    int n_sph_nl, n_fin_nl, n_inf_nl;   // non-light prefix lengths
    int n_sph_bvh, n_fin_bvh;           // BVH-covered prefix of the non-light prefix (0 = none)
    int n_lights;
    int fin_off, inf_off, light_off, idx_off;   // float4 offsets into the blob
    // finite-plane array order: [generic non-light | axis-aligned ("arect", never lights) | lights];
    // arects are reached through the box clusters only.  n_fin_gen == n_fin_nl - n_arect.
    int n_fin_gen, n_arect;
    int n_clu, clu_off, cslot_off;
    float clu_cx, clu_cy, clu_cz, clu_rbig;   // hull centre of the clusters; L1 radius + largest |coordinate|
    // winner-only, indexed by object index
    const float4* obj_surface;   // colour rgb, diffuse
    const float4* obj_material;  // specular, reflective, intensity, 0
    const float4* obj_normals;   // 6 per object: (n1, normalize(n1), normalize^2(n1)) facing, then reverse
    const int4* obj_info;        // type, slot (position in the permuted type array), is_light, texture id
    const float4* inf_frame;     // 3 per infinite plane slot: horizontal, vertical, origin
    const float4* textures;      // 2 per texture: (light rgb, width) (dark rgb, height)
    // optional BVHs over the non-light spheres / finite planes (nullptr = linear sweep); the
    // type's primitive array is then in leaf order.  Node layout: see tcrt_render.cu.
    const float4* bvh_sph;
    const float4* bvh_fin;
    int bvh_sph_root, bvh_fin_root;   // encoded like a child reference
    // optional uniform grid over the BVH-covered spheres (nullptr = none): a 3D-DDA finds the cells a ray crosses,
    // the spheres registered in a cell are tested exactly.  Rays fattened by more than grid_margin use the BVH.
    const float4* grid_cells;         // 2 per cell: (geometry of the cell's first sphere; r^2 = -1e30 in an empty cell: never
                                      // hit) (number of FURTHER spheres, slot of the first sphere, position of the second one
                                      // in grid_items, -) — the usual cell holds one sphere and costs ONE round of loads
    const int* grid_items;            // sphere slots, cell after cell
    float grid_lo[3], grid_hi[3], grid_cell[3], grid_inv_cell[3];   // hi = lo + cell * dims
    int grid_dims[3];
    float grid_margin;
    float grid_k2_max;                // fatten().m <= grid_margin  <=>  its k2 <= grid_k2_max (m grows with k2)
    // per-ray fattening of the boxes (tcrt_render.cu `fatten`): bounding sphere (centre, radius^2)
    // of everything inside the BVHs, smallest BVH sphere radius, largest |coordinate|
    float bvh_cx, bvh_cy, bvh_cz, bvh_r2, bvh_rmin, bvh_cmax;
};

// host BVH builder (tcrt_bvh.cpp).  boxes: n x 6 floats (lo xyz, hi xyz), already inflated.
// On return `order` is the leaf order (a permutation of 0..n-1), `nodes` 4 float4 per node,
// and the function value is the encoded root reference.
#ifdef __cplusplus
#include <vector>
int tcrt_build_bvh(const std::vector<float>& boxes, int n, std::vector<int>& order, std::vector<float4>& nodes,
                   int* depth);   // *depth: deepest node; the kernel's traversal stack holds TCRT_BVH_STACK entries
#define TCRT_BVH_STACK 48
// E = TCRT_SPH_E * 2(|O - Cs|^2 + Rs^2) bounds the rounding of the reference's sphere discriminant (`fatten`,
// tcrt_render_common.cuh); the host derives the grid's far-origin bound from the same constant
#define TCRT_SPH_E 4e-6f

// host builder of the uniform grid over the BVH-covered spheres (tcrt_bvh.cpp)
struct TcrtSphereGrid {
    float lo[3] = {0, 0, 0};
    float cell[3] = {1, 1, 1};
    int dims[3] = {0, 0, 0};
    float reg_margin = 0.f;             // a ray whose fattening is below this may use the grid
    std::vector<int> cell_start;        // dims[0]*dims[1]*dims[2] + 1
    std::vector<int> items;             // sphere slots (leaf order), cell by cell
};
bool tcrt_build_sphere_grid(const std::vector<float>& boxes, int n, TcrtSphereGrid& g);
#endif

// Pixel tile of one queue claim: TCRT_TILE_W columns x TCRT_TILE_H rows = 32 pixels, one per lane.
#ifndef TCRT_TILE_W
#define TCRT_TILE_W 4
#endif
#define TCRT_TILE_H (32 / TCRT_TILE_W)

struct RenderLaunch {
    DeviceScene scene;
    tcrt_camera cam;
    int width, height;
    int x0, x1;              // columns rendered by this launch
    int max_depth;
    int shadows_on, reflections_on;
    float null_r, null_g, null_b;
    float far_dist;
    float* out;              // (x1-x0)*height*3 floats, x-major
    unsigned int* queue;     // pixel queue head (zeroed before launch)
    unsigned long long* counters;   // [0] primary [1] shadow [2] reflect
    const int* row_order;    // optional: permutation of the rows [0, height) — of the 8-row tile rows [0, height/8) when
                             // `tiled` — in which the queue runs
    unsigned int* col_cost;  // optional (balancer pre-pass): [x1-x0] per column then [height] per row, += bounces of every finished pixel
    int n_objects;           // objects of the scene (checked builds verify table indices against it)
    int refill_min;          // idle lanes a warp waits for before it takes new pixels (1..32)
    int tiled;               // queue positions map to 4x8-pixel tiles (band width % 4 == 0, height % 8 == 0)
    int prune_dead;          // every colour the reference forms is finite: the grid kernel may skip the shading of levels
                             // whose contribution is multiplied by a zero object colour (dead_path_bound, tcrt_api.cu)
    // list mode (tcrt_launch_render_list, adaptive frames): width x height is the ss*W x ss*H sample frame, x0 == 0, and
    // queue position q traces sample 1 + q % (ss*ss-1) of frame pixel list[q / (ss*ss-1)] (x*H + z of the W x H frame)
    // into out[3q..3q+2] (list_to_sample, tcrt_render_common.cuh).  Band mode ignores these.
    const int* list;
    int list_n;              // queue positions: list entries * (ss*ss - 1); in ray mode the rays of the launch
    int list_ss;
    // ray mode (tcrt_launch_render_rays, ray batches): queue position q traces the caller's ray q — origin
    // ray_o[ray_o_stride*q ..], direction ray_d[3q ..] — into out[3q..3q+2], x0 == 0 and the camera unused.  A ray that
    // fails the validity rule of tcrt.h (ray_from_batch, tcrt_render_common.cuh) is not traced: out gets quiet NaNs and
    // *ray_invalid counts it.  The other modes ignore these.
    const float* ray_o;
    int ray_o_stride;        // 3, or 0: one origin shared by every ray
    const float* ray_d;
    unsigned long long* ray_invalid;
};

// What a render launch traces: the pixels of a band, the samples of a pixel list, or a batch of caller-supplied rays.
// A compile-time parameter of the render kernel bodies (one kernel per mode keeps each bounce loop in the instruction cache).
enum RenderMode { kModeBand = 0, kModeList = 1, kModeRays = 2 };

// Primary-hit launch (tcrt_hits.cu): rl describes the frame, the band [x0, x1) and the scene; out of rl the kernel uses the
// camera, width, height, x0, x1, far_dist, queue and n_objects.  Band mode (xz == nullptr): every pixel of the band, x-major
// like frames.  List mode: entry i is pixel (xz[2i], xz[2i+1]) of the frame (rl.x0 == 0), and output i is its hit.
// Ray mode (rl.ray_d != nullptr): output i is the hit of ray i of the batch, rl.list_n rays, with rl's ray fields as in
// render ray mode; an invalid ray gets object -2, distance and normal NaN.  Each output pointer may be nullptr there.
struct HitLaunch {
    RenderLaunch rl;
    const int* xz;
    int n_list;
    int* object;       // per pixel: object index of the nearest hit, -1 on a miss
    float* distance;   // its distance (far_dist on a miss)
    float* normal;     // 3 per pixel: its normal ray's direction ((0,0,0) on a miss)
};

// Occlusion launch (tcrt_hits.cu, tcrt_occluded_rays / tcrt_occluded_lights): the shadow test of inShadeCollisionDetection
// for rl.list_n items.  Out of rl the kernel uses the scene, queue, counters[1] (tests traced), ray_invalid (invalid rays or
// pairs) and n_objects.  Rays mode (points == nullptr): item q is ray q of rl's ray fields (render ray mode) with limit
// tmax[q], answered in out[q].  Points mode: item q is the point points[3q..3q+2], tested against every light l of the
// scene along the reference's inShade construction, answered in out[q * n_lights + l].  An answer is 1 (occluded), 0, or
// 0xFF for an invalid ray or pair.
struct OccLaunch {
    RenderLaunch rl;
    const float* tmax;
    const float* points;
    unsigned char* out;
};

// host builder of the box clusters (tcrt_cluster.cpp).  Face f = 2*axis + k; an absent face has
// c = NaN and plane = -1; `plane` indexes the caller's list.
struct TcrtBoxCluster {
    float lo[3], hi[3];
    float c[6];
    int plane[6];
};
#ifdef __cplusplus
// planes: indices into fin_geom (16 floats each) of the candidate (non-light) finite planes.
// arect_of_plane[i] != 0 when planes[i] is axis-aligned and therefore owned by a cluster.
void tcrt_build_box_clusters(const float* fin_geom, const std::vector<int>& planes, std::vector<int>& arect_of_plane,
                             std::vector<TcrtBoxCluster>& out);
#endif

// render kernels (tcrt_render.cu).  wave_mem / wave_bytes: scratch for the wavefront path (tcrt_render_wave.cu), which
// tcrt_launch_render takes for large frames of sphere-BVH scenes when the scratch is big enough (tcrt_wave_mem_needed).
cudaError_t tcrt_launch_render(const RenderLaunch& rl, int sm_count, cudaStream_t stream, int* launches, void* wave_mem,
                               size_t wave_bytes);
// bytes of scratch the wavefront path wants for this launch, 0 when the launch does not take that path
size_t tcrt_wave_mem_needed(const RenderLaunch& rl);
bool tcrt_wave_applies(const RenderLaunch& rl, int fm);
size_t tcrt_wave_mem_bytes(size_t band_pixels, int max_depth);
cudaError_t tcrt_launch_render_wave(const RenderLaunch& rl, int fm, int sm_count, size_t smem_scene, void* mem, size_t mem_bytes,
                                    cudaStream_t stream, int* launches);
size_t tcrt_render_max_smem();
// kernel for scenes whose spheres sit in a uniform grid (tcrt_render_grid.cu); smem = bytes of the staged blob
cudaError_t tcrt_launch_render_grid(const RenderLaunch& rl, int fm, int sm_count, size_t smem, cudaStream_t stream,
                                    RenderMode mode = kModeBand);
// list-mode render launch (adaptive frames, RenderLaunch::list): the render or grid kernel's list-mode twin, one launch
cudaError_t tcrt_launch_render_list(const RenderLaunch& rl, int sm_count, cudaStream_t stream);
// ray-mode render launch (ray batches, RenderLaunch::ray_*): the render or grid kernel's ray-mode twin, one launch of
// rl.list_n rays; nothing when there are none
cudaError_t tcrt_launch_render_rays(const RenderLaunch& rl, int sm_count, cudaStream_t stream);
// experimental task-pool kernel for sphere-BVH scenes (tcrt_render_pool.cu, developer builds only); smem_scene = bytes of the staged blob
cudaError_t tcrt_launch_render_pool(const RenderLaunch& rl, int fm, int sm_count, size_t smem_scene, cudaStream_t stream);
// n random (a.xyz, b) cases: div3 (shared-reciprocal division of the render kernel) vs __fdiv_rn; *bad += mismatches
cudaError_t tcrt_launch_div3_check(unsigned long long n, unsigned seed, unsigned long long* bad, cudaStream_t stream);   // dynamic shared memory the kernel may opt in to

// primary-hit buffers and picks (tcrt_hits.cu): one launch, nothing when there are no pixels
cudaError_t tcrt_launch_hits(const HitLaunch& hl, int sm_count, cudaStream_t stream);
// occlusion queries (tcrt_hits.cu): one launch, nothing when there are no items
cudaError_t tcrt_launch_occlusion(const OccLaunch& ol, int sm_count, cudaStream_t stream);

// txt formatter (tcrt_format.cu)
// fixed path: 31-byte lines; general path: per-pixel lengths -> two-level exclusive scan
// (offs: n_pixels uint64 tile-local offsets; block_sums: ceil(n/256)+1 uint64, last = total).
cudaError_t tcrt_launch_txt_fixed_check(const float* rgb, size_t n_pixels, unsigned int* not_fixed_flag,
                                        cudaStream_t stream);
cudaError_t tcrt_launch_txt_fixed(const float* rgb, size_t n_pixels, char* text, cudaStream_t stream);
cudaError_t tcrt_launch_txt_lengths(const float* rgb, size_t n_pixels, unsigned long long* offs,
                                    unsigned long long* block_sums, cudaStream_t stream, int* launches);
cudaError_t tcrt_launch_txt_general(const float* rgb, size_t n_pixels, const unsigned long long* offs,
                                    const unsigned long long* block_offs, char* text, cudaStream_t stream);
// 8-bit quantisation + transposition of an x-major band (cols x height) into image rows (top row first, cols pixels each)
cudaError_t tcrt_launch_quantize8_image(const float* rgb, int cols, int height, unsigned char* out, cudaStream_t stream);
// 8-bit quantisation in place order (the RGB8 frames of tcrt_render_rgb8): byte j of out = q(rgb[j]), j < 3*n_pixels.
// Any start address of either buffer.
cudaError_t tcrt_launch_quantize8(const float* rgb, size_t n_pixels, unsigned char* out, cudaStream_t stream);
// Supersampled frames (tcrt_render_columns_ss): cols x height output pixels, x-major, each the mean of its ss x ss samples
// in `samples` (ss*cols x ss*height sample pixels, x-major, 1 <= ss <= 8) summed in the order of tcrt.h; out8 (nullable)
// gets the same pixels quantised to 8 bits in the same pass.  samples must be 16-byte aligned.
cudaError_t tcrt_launch_resolve_ss(const float* samples, int cols, int height, int ss, float* out, unsigned char* out8,
                                   cudaStream_t stream);
// Adaptive frames (tcrt_adaptive.cu).  classify: for band [bx0, bx1) of the width x height frame, from the plain frame's
// columns [px0, ...) (the band and its in-frame halo columns): mask[p] (1 = refined, contrast < 0 refines every pixel),
// frame[p] = the plain pixel, then the refined pixels' x*height + z, x-major, into list and their number into
// block_counts[ceil(band pixels / 256)] (block_counts holds that many + 1 words).  Three launches.
cudaError_t tcrt_launch_adaptive_classify(const float* plain, int px0, int width, int height, int bx0, int bx1, int contrast,
                                          float* frame, unsigned char* mask, unsigned int* block_counts, int* list,
                                          cudaStream_t stream);
// resolve of list entries [e0, e0 + n): samples 1 .. ss*ss-1 of entry e0 + t are scratch[(t*(ss*ss-1) + s-1)*3 ..] (the
// list-mode render launch's output), sample 0 is the band's frame pixel; the mean, in tcrt.h's order, replaces it.
cudaError_t tcrt_launch_adaptive_resolve(const int* list, int e0, int n, int bx0, int height, int ss, const float* scratch,
                                         float* frame, cudaStream_t stream);
cudaError_t tcrt_launch_l2_flush(void* scratch, size_t bytes, cudaStream_t stream);
// 8 independent chains per thread, `iters` rounds: 8*iters FFMA, or 8*iters FMUL + 8*iters FADD
cudaError_t tcrt_launch_fp32_peak(bool fma, float* scratch, int grid, int iters, cudaStream_t stream);

#endif  // TCRT_DEVICE_H_
