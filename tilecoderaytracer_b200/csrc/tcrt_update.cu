// tcrt_update.cu — moving spheres (tcrt_update_spheres): the resident scene's spheres take new centres and radii in place,
// and the pruning structures follow them on the device, without the host's sort, SAH build and grid search.  Moving planes
// (tcrt_update_planes) scatter the rows the host planned and refit the finite-plane BVH with the same refit launch.
//
// Every structure only decides WHICH primitives a ray tests; the tests themselves are the reference's arithmetic
// (DESIGN.md §4.5).  So a BVH keeps its topology and leaf order and only has its boxes refitted around the moved spheres,
// and the sphere grid keeps its origin, cell size and dimensions and has its cells registered again with the builder's
// own arithmetic (tcrt_build_sphere_grid).  Both stay sound; the host drops the grid when a sphere's widened box leaves
// the grid's box or the registrations break the builder's acceptance rules (UpdateBack::grid_out, grid_full).
//
// Launches, all on the render stream: (1) validate every sphere and reduce the scene-wide maxima; (2) scatter each sphere
// into its blob slot, box the BVH's spheres as the upload does (sphere_box, tcrt_api.cu) and count their grid
// registrations; (3) refit the BVH level by level in one block; (4) scan the counts, emit (cell, sphere) pairs, sort them
// by cell (stable: a cell lists its spheres in increasing leaf order, as the builder writes them) into scratch, scan the
// cell counts, and rewrite every cell record and the item list from the scratch.  Launches after (1) write nothing the scene
// reads when the input is invalid: the scans and the sort work in scratch buffers, and only the last launch, which checks
// the flags first, writes the cells and the item list.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

#include "tcrt_device.h"

namespace {

constexpr int kUpdBlock = 256;
constexpr int kRefitBlock = 1024;

// order-preserving map of a finite float onto unsigned (atomicMax / atomicMin of floats of either sign)
__device__ __forceinline__ unsigned order_key(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__device__ __forceinline__ bool sphere_ok(float4 g) {
    return isfinite(g.x) && isfinite(g.y) && isfinite(g.z) && isfinite(g.w) && g.w >= 0.0f;
}

// the upload's ext: max(1, |finite-plane origins|, |sphere centres|), 1e30 when not finite (plan_scene_blob)
__device__ __forceinline__ double update_ext(const UpdateLaunch& ul) {
    double ext = fmax(ul.ext_fixed, (double)__uint_as_float(ul.back->ext_bits));
    return isfinite(ext) ? ext : 1e30;
}

// (1) validity, max |centre component|, smallest radius_squared over the BVH's spheres, the light spheres' centres
__global__ void __launch_bounds__(kUpdBlock) update_reduce_kernel(const UpdateLaunch ul) {
    const int i = blockIdx.x * kUpdBlock + threadIdx.x;
    unsigned bad = 0u, ext = 0u, r2key = 0u;
    if (i < ul.n) {
        const float4 g = ul.geom[i];
        bad = sphere_ok(g) ? 0u : 1u;
        ext = __float_as_uint(fmaxf(fmaxf(fabsf(g.x), fabsf(g.y)), fabsf(g.z)));
        if (ul.slot_of[i] < ul.n_bvh) r2key = ~__float_as_uint(g.w + 0.0f);   // + 0: -0 -> +0
    }
    bad = __reduce_or_sync(0xffffffffu, bad);
    ext = __reduce_max_sync(0xffffffffu, ext);
    r2key = __reduce_max_sync(0xffffffffu, r2key);
    if ((threadIdx.x & 31) == 0) {
        if (bad) atomicOr(&ul.back->invalid, 1u);
        atomicMax(&ul.back->ext_bits, ext);
        if (r2key) atomicMax(&ul.back->r2min_key, r2key);
    }
    if (i < ul.n_light_sph) {
        const float4 g = ul.geom[ul.light_sph[i]];
        float* pos = reinterpret_cast<float*>(ul.back + 1) + 3 * i;
        pos[0] = g.x;
        pos[1] = g.y;
        pos[2] = g.z;
    }
}

// The grid cells [a, b] per axis of a box, with the builder's arithmetic; false when the widened box leaves the grid
__device__ __forceinline__ bool grid_range(const UpdateLaunch& ul, const float* box, int* a, int* b) {
    bool inside = true;
    for (int k = 0; k < 3; k++) {
        const double fa = floor(((double)box[k] - ul.gmargin - ul.glo[k]) / ul.gcell[k]);
        const double fb = floor(((double)box[3 + k] + ul.gmargin - ul.glo[k]) / ul.gcell[k]);
        inside = inside && fa >= 0.0 && fb <= (double)(ul.gdims[k] - 1);
        a[k] = (int)fmin(fmax(fa, 0.0), (double)(ul.gdims[k] - 1));
        b[k] = (int)fmin(fmax(fb, 0.0), (double)(ul.gdims[k] - 1));
    }
    return inside;
}

// (2) scatter, boxes and their bounds, grid registration counts
__global__ void __launch_bounds__(kUpdBlock) update_scatter_kernel(const UpdateLaunch ul) {
    if (ul.back->invalid) return;
    const int i = blockIdx.x * kUpdBlock + threadIdx.x;
    if (i >= ul.n) return;
    const float4 g = ul.geom[i];
    const int slot = ul.slot_of[i];
    ul.spheres[slot] = g;
    if (slot >= ul.n_boxed) return;
    // sphere_box (tcrt_api.cu) in the same double arithmetic (this file is built with -fmad=false)
    const double margin = 1e-5 * update_ext(ul);
    const double r = sqrt(fmax(0.0, (double)g.w)) * (1.0 + 1e-6);
    const float c[3] = {g.x, g.y, g.z};
    float box[6];
    for (int k = 0; k < 3; k++) {
        box[k] = (float)((double)c[k] - r - margin - 1e-6 * fabs((double)c[k]));
        box[3 + k] = (float)((double)c[k] + r + margin + 1e-6 * fabs((double)c[k]));
        if (isfinite(box[k])) atomicMax(&ul.back->lo_key[k], ~order_key(box[k]));
        if (isfinite(box[3 + k])) atomicMax(&ul.back->hi_key[k], order_key(box[3 + k]));
    }
    float* out = ul.boxes + 6 * (size_t)slot;
    for (int k = 0; k < 6; k++) out[k] = box[k];
    if (ul.grid && slot < ul.n_bvh) {
        int a[3], b[3];
        if (!grid_range(ul, box, a, b)) atomicOr(&ul.back->grid_out, 1u);
        ul.reg_count[slot] = (unsigned)(b[0] - a[0] + 1) * (unsigned)(b[1] - a[1] + 1) * (unsigned)(b[2] - a[2] + 1);
    }
}

// (3) the sphere BVH's boxes, deepest level first: a node holds the boxes of its two children (tcrt_bvh.cpp), a leaf's box
// is the union of its spheres' boxes, an inner child's the union of the two boxes it holds
__device__ __forceinline__ void child_box(const UpdateLaunch& ul, int ref, float* bx) {
    for (int k = 0; k < 3; k++) {
        bx[k] = INFINITY;
        bx[3 + k] = -INFINITY;
    }
    if (ref < 0) {
        const int v = ~ref, first = v & 0xffffff, last = first + (v >> 24);
        for (int s = first; s < last; s++)
            for (int k = 0; k < 3; k++) {
                bx[k] = fminf(bx[k], ul.boxes[6 * (size_t)s + k]);
                bx[3 + k] = fmaxf(bx[3 + k], ul.boxes[6 * (size_t)s + 3 + k]);
            }
    } else {
        const float4 a = ul.nodes[4 * ref], b = ul.nodes[4 * ref + 1], c = ul.nodes[4 * ref + 2];
        const float lo0[3] = {a.x, a.y, a.z}, hi0[3] = {a.w, b.x, b.y}, lo1[3] = {b.z, b.w, c.x}, hi1[3] = {c.y, c.z, c.w};
        for (int k = 0; k < 3; k++) {
            bx[k] = fminf(lo0[k], lo1[k]);
            bx[3 + k] = fmaxf(hi0[k], hi1[k]);
        }
    }
}

__global__ void __launch_bounds__(kRefitBlock) update_refit_kernel(const UpdateLaunch ul) {
    if (ul.back->invalid) return;
    for (int l = ul.n_levels - 1; l >= 0; l--) {
        for (int j = ul.level_start[l] + threadIdx.x; j < ul.level_start[l + 1]; j += kRefitBlock) {
            const int node = ul.levels[j];
            const float4 ch = ul.nodes[4 * node + 3];
            float b0[6], b1[6];
            child_box(ul, __float_as_int(ch.x), b0);
            child_box(ul, __float_as_int(ch.y), b1);
            ul.nodes[4 * node + 0] = make_float4(b0[0], b0[1], b0[2], b0[3]);
            ul.nodes[4 * node + 1] = make_float4(b0[4], b0[5], b1[0], b1[1]);
            ul.nodes[4 * node + 2] = make_float4(b1[2], b1[3], b1[4], b1[5]);
        }
        __syncthreads();   // the next level up reads these nodes (global memory, one block)
    }
}

// (4a) one (cell, slot) pair per registration, sphere after sphere; the unused tail of the buffer sorts last
__global__ void __launch_bounds__(kUpdBlock) update_emit_kernel(const UpdateLaunch ul) {
    const unsigned long long* off = ul.reg_off;
    const unsigned long long total = off[ul.n_bvh];
    const bool ok = !ul.back->invalid && !ul.back->grid_out && total <= ul.cap;
    if (blockIdx.x == 0 && threadIdx.x == 0 && total > ul.cap) atomicOr(&ul.back->grid_full, 1u);
    const unsigned i = blockIdx.x * kUpdBlock + threadIdx.x;
    if (i < ul.cap && (!ok || i >= total)) {
        ul.keys[i] = (unsigned)ul.n_cells;
        ul.vals[i] = 0u;
    }
    if (!ok || i >= (unsigned)ul.n_bvh) return;
    int a[3], b[3];
    grid_range(ul, ul.boxes + 6 * (size_t)i, a, b);
    unsigned q = (unsigned)off[i];
    for (int z = a[2]; z <= b[2]; z++)
        for (int y = a[1]; y <= b[1]; y++)
            for (int x = a[0]; x <= b[0]; x++) {
                const unsigned c = (unsigned)x + (unsigned)ul.gdims[0] * ((unsigned)y + (unsigned)ul.gdims[1] * (unsigned)z);
                ul.keys[q] = c;
                ul.vals[q] = i;
                q++;
                atomicAdd(&ul.cell_count[c], 1u);
            }
}

// (4b) the item list, copied from the sort's scratch, and the cell records (tcrt_api.cu plan_scene_blob): the first
// sphere's geometry, then (further spheres, first slot, position of the second one in the item list, 0); an empty cell
// carries a sphere no ray hits.  Nothing is written after a failed check.  A cell of more than 24 spheres is found here,
// while other threads write: the host then drops the grid, so no launch reads what was written.
__global__ void __launch_bounds__(kUpdBlock) update_cells_kernel(const UpdateLaunch ul) {
    if (ul.back->invalid || ul.back->grid_out || ul.back->grid_full) return;
    const unsigned t = blockIdx.x * kUpdBlock + threadIdx.x;
    if (t < ul.cap) ul.items[t] = (int)ul.sorted[t];
    const int c = (int)t;
    if (c >= ul.n_cells) return;
    const unsigned cnt = ul.cell_count[c], j0 = ul.cell_start[c];
    if (cnt > 24u) atomicOr(&ul.back->grid_full, 1u);
    const int first = cnt > 0u ? (int)ul.sorted[j0] : 0;
    ul.cells[2 * c] = cnt > 0u ? ul.spheres[first] : make_float4(0.f, 0.f, 0.f, -1e30f);
    const int4 meta = make_int4(cnt > 0u ? (int)cnt - 1 : 0, first, (int)j0 + 1, 0);
    reinterpret_cast<int4*>(ul.cells)[2 * c + 1] = meta;
}

// Moving planes (tcrt_update_planes): every row the host planned for the moved scene, written into the blob
__global__ void __launch_bounds__(kUpdBlock) plane_scatter_kernel(const PlaneLaunch pl) {
    const int i = blockIdx.x * kUpdBlock + threadIdx.x;
    if (i >= pl.n) return;
    const PlaneRecord r = pl.rec[i];
    pl.scene[r.dst] = r.v;
}

int key_bits(int n_cells) {   // bits of the keys 0 .. n_cells (n_cells: the tail's key)
    int b = 1;
    while ((1u << b) <= (unsigned)n_cells && b < 32) b++;
    return b;
}

}  // namespace

size_t tcrt_update_tmp_bytes(unsigned cap, int n_bvh, int n_cells) {
    size_t a = 0, b = 0, c = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, a, (unsigned long long*)nullptr, (unsigned long long*)nullptr, n_bvh + 1);
    cub::DeviceRadixSort::SortPairs(nullptr, b, (unsigned*)nullptr, (unsigned*)nullptr, (unsigned*)nullptr, (unsigned*)nullptr,
                                    (int)cap, 0, key_bits(n_cells));
    cub::DeviceScan::ExclusiveSum(nullptr, c, (unsigned*)nullptr, (unsigned*)nullptr, n_cells + 1);
    return std::max(a, std::max(b, c));
}

cudaError_t tcrt_launch_update_spheres(const UpdateLaunch& ul, int sm_count, cudaStream_t stream, int* launches) {
    (void)sm_count;
    if (ul.n <= 0) return cudaSuccess;
    const int blocks = (ul.n + kUpdBlock - 1) / kUpdBlock;
    const int light_blocks = (ul.n_light_sph + kUpdBlock - 1) / kUpdBlock;
    cudaError_t e = cudaMemsetAsync(ul.back, 0, sizeof(UpdateBack) + 12 * (size_t)ul.n_light_sph, stream);
    if (e == cudaSuccess && ul.grid) e = cudaMemsetAsync(ul.reg_count, 0, 8 * ((size_t)ul.n_bvh + 1), stream);
    if (e == cudaSuccess && ul.grid) e = cudaMemsetAsync(ul.cell_count, 0, 4 * ((size_t)ul.n_cells + 1), stream);
    if (e != cudaSuccess) return e;
    update_reduce_kernel<<<std::max(blocks, light_blocks), kUpdBlock, 0, stream>>>(ul);
    update_scatter_kernel<<<blocks, kUpdBlock, 0, stream>>>(ul);
    *launches += 2;
    if (ul.n_levels > 0) {
        update_refit_kernel<<<1, kRefitBlock, 0, stream>>>(ul);
        *launches += 1;
    }
    if ((e = cudaGetLastError()) != cudaSuccess || !ul.grid) return e;
    size_t tmp = ul.tmp_bytes;
    e = cub::DeviceScan::ExclusiveSum(ul.tmp, tmp, ul.reg_count, ul.reg_off, ul.n_bvh + 1, stream);
    if (e != cudaSuccess) return e;
    update_emit_kernel<<<(std::max<unsigned>(ul.cap, (unsigned)ul.n_bvh) + kUpdBlock - 1) / kUpdBlock, kUpdBlock, 0, stream>>>(ul);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    tmp = ul.tmp_bytes;
    e = cub::DeviceRadixSort::SortPairs(ul.tmp, tmp, ul.keys, ul.keys2, ul.vals, ul.sorted, (int)ul.cap, 0, key_bits(ul.n_cells),
                                        stream);
    if (e != cudaSuccess) return e;
    tmp = ul.tmp_bytes;
    e = cub::DeviceScan::ExclusiveSum(ul.tmp, tmp, ul.cell_count, ul.cell_start, ul.n_cells + 1, stream);
    if (e != cudaSuccess) return e;
    update_cells_kernel<<<(std::max<unsigned>(ul.cap, (unsigned)ul.n_cells) + kUpdBlock - 1) / kUpdBlock, kUpdBlock, 0, stream>>>(ul);
    *launches += 5;   // the scans and the sort count as one launch each
    return cudaGetLastError();
}

cudaError_t tcrt_launch_update_planes(const PlaneLaunch& pl, cudaStream_t stream, int* launches) {
    if (pl.n > 0) {
        plane_scatter_kernel<<<(pl.n + kUpdBlock - 1) / kUpdBlock, kUpdBlock, 0, stream>>>(pl);
        *launches += 1;
    }
    if (pl.n_levels > 0) {   // the finite-plane BVH, refitted like the sphere BVH from its leaves' boxes (slots = leaf order)
        UpdateLaunch ul{};
        ul.back = pl.back;
        ul.boxes = const_cast<float*>(pl.boxes);   // read only
        ul.nodes = pl.nodes;
        ul.levels = pl.levels;
        ul.level_start = pl.level_start;
        ul.n_levels = pl.n_levels;
        cudaError_t e = cudaMemsetAsync(pl.back, 0, sizeof(UpdateBack), stream);
        if (e != cudaSuccess) return e;
        update_refit_kernel<<<1, kRefitBlock, 0, stream>>>(ul);
        *launches += 1;
    }
    return cudaGetLastError();
}
