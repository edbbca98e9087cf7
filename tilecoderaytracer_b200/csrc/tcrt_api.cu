// tcrt_api.cu — the C ABI of include/tcrt.h: contexts, scene upload, render launches,
// copy-back, the .txt writer.  No CPU render path exists here: without a CUDA device every
// entry point that needs one fails.
#include <errno.h>
#include <fcntl.h>
#include <stdarg.h>
#include <unistd.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <limits.h>

#include <math.h>

#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/vfs.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "tcrt_device.h"

namespace {

// What one frame in flight owns on a device.  Two sets per device: tcrt_render_async renders frame n+1 into one
// while frame n's band is still being copied out of the other.
constexpr int kMaxChunks = 16;     // column chunks of a band that goes to host memory (= events per frame)
#ifndef TCRT_CHUNK_STREAMS
#define TCRT_CHUNK_STREAMS 4
#endif
constexpr int kChunkStreams = TCRT_CHUNK_STREAMS;   // streams their launches alternate on

struct FrameRes {
    float* frame = nullptr;                   // the band, (x1-x0)*height*3 floats, x-major
    size_t frame_cap = 0;                     // floats
    unsigned char* frame8 = nullptr;          // the band quantised to 8 bits, (x1-x0)*height*3 bytes, x-major (RGB8 frames)
    size_t frame8_cap = 0;                    // bytes
    int x0 = 0, x1 = 0, height = 0;
    unsigned char* ctl = nullptr;             // queue head @0, ray counters @8..31, queue heads of the column chunks @64 (kMaxChunks x u32)
    unsigned long long* h_counters = nullptr; // pinned, 4 x u64 (slot 0 unused)
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;   // around the kernels (render stream)
    cudaEvent_t ev_done = nullptr;            // ray counters are in h_counters (render stream)
    cudaEvent_t ev_c1 = nullptr;              // last chunk is in host memory (copy stream)
    cudaEvent_t ev_chunk[kMaxChunks] = {};            // chunk k rendered
    cudaEvent_t ev_start = nullptr;           // control block zeroed, row order uploaded (render stream)
    int n_chunks = 0, chunk_x[kMaxChunks + 1] = {};   // the column chunks of the frame being rendered (ev_chunk[k] covers [chunk_x[k], chunk_x[k+1]))
};

struct DeviceState {
    int dev = -1;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t chunk_stream[kChunkStreams - 1] = {};   // with `stream`: the column chunks of a band that goes to host memory, round robin (render_submit)
    cudaStream_t copy_stream = nullptr;           // D2H of finished column chunks, behind the render streams
    // scene
    float4* scene_mem = nullptr;
    size_t scene_cap_f4 = 0;
    DeviceScene ds{};
    cudaEvent_t ev_scene = nullptr;               // the last scene upload has left its pinned staging buffer
    // frames
    FrameRes res[2];
    int cur = 0;                                  // the set the synchronous API (and the last waited-for frame) uses
    FrameRes& fr() { return res[cur]; }
    // txt scratch
    char* text = nullptr;
    size_t text_cap = 0;
    unsigned long long* offs = nullptr;
    size_t offs_cap = 0;
    unsigned long long* block_sums = nullptr;
    size_t bs_cap = 0;
    unsigned int* flag = nullptr;             // device, 16 B
    unsigned long long* h_txt = nullptr;      // pinned: [0] flag, [1] total bytes
    bool txt_fixed = true;
    size_t txt_bytes = 0;
    char* txt_stage = nullptr;                // pinned: kTxtSlots chunks of text on their way to the file (tcrt_write_txt)
    cudaEvent_t ev_txt[4] = {};               // chunk in staging slot k has arrived
    // row order of the current launch (most expensive rows first)
    int* row_order = nullptr;
    size_t row_order_cap = 0;
    unsigned long long row_order_serial = 0;
    int row_order_h = 0;
    // balancer pre-pass: bounce counts per column, then per row (tcrt_balance_columns)
    unsigned int* col_cost = nullptr;
    size_t col_cost_cap = 0;
    // wavefront scratch (tcrt_render_wave.cu)
    void* wave_mem = nullptr;
    size_t wave_bytes = 0;
    // L2 flush scratch
    void* flush = nullptr;
    size_t flush_bytes = 0;
    // supersampled frames: the sample columns of one column chunk, one buffer per render stream (0 = `stream`, then
    // chunk_stream[]).  The chunk's render launch and its resolve launch run on that stream, and so does every later
    // chunk that reuses the buffer, so both frame sets share it.
    float* ss_scratch[kChunkStreams] = {};
    size_t ss_scratch_cap[kChunkStreams] = {};     // floats
    // primary-hit buffers (tcrt_hit_buffers) and picks (tcrt_pick): buffers, queue head and events of their own, so that
    // neither touches the last render or a frame in flight.  hit_mem holds the band of the last tcrt_hit_buffers call:
    // n = (hit_x1 - hit_x0) * hit_h object indices, then n distances, then 3n normal components.  pick_mem: the 2n
    // coordinates of a pick, then its 5n result words in the same layout.
    float* hit_mem = nullptr;
    size_t hit_mem_cap = 0;                       // 4-byte words
    int hit_x0 = 0, hit_x1 = 0, hit_h = 0;
    int* pick_mem = nullptr;
    size_t pick_mem_cap = 0;                      // 4-byte words
    unsigned int* hit_queue = nullptr;            // device, 16 B
    cudaEvent_t ev_h0 = nullptr, ev_h1 = nullptr; // around the hit kernel (render stream)
    cudaEvent_t ev_hc = nullptr;                  // the direct copies of the hit buffers are in host memory (copy stream)
    // adaptive frames (tcrt_render_columns_adaptive): the plain frame over the band and its halo columns, the band's mask,
    // the classify pass's per-CTA counts (then their exclusive scan and the total), the list of refined pixels.  The call
    // is synchronous: nothing else uses them while it runs.
    float* ad_plain = nullptr;
    size_t ad_plain_cap = 0;                      // floats
    unsigned char* ad_mask = nullptr;
    size_t ad_mask_cap = 0;
    unsigned int* ad_counts = nullptr;
    size_t ad_counts_cap = 0;
    int* ad_list = nullptr;
    size_t ad_list_cap = 0;
    // ray batches (tcrt_trace_rays, tcrt_intersect_rays): per render stream the device scratch of one piece (its inputs,
    // then its outputs) and the pinned staging of pageable inputs, allocated at first use; queue heads, counters and
    // events of their own, so that a batch touches neither the last render nor a frame in flight.  The calls are
    // synchronous: nothing else uses these while one runs.
    float* ray_mem[kChunkStreams] = {};
    size_t ray_mem_cap[kChunkStreams] = {};        // floats
    float* ray_stage[kChunkStreams] = {};
    size_t ray_stage_cap[kChunkStreams] = {};      // floats
    unsigned char* ray_ctl = nullptr;              // 64 B per render stream: queue head @0, ray counters @8..31, invalid @32
    unsigned long long* h_ray = nullptr;           // pinned copy of ray_ctl
    cudaEvent_t ev_r0 = nullptr, ev_r1 = nullptr;  // first input copy / last launch done (render stream)
    cudaEvent_t ev_rc = nullptr;                   // the last output copy is in host memory (copy stream)
    cudaEvent_t ev_rk[kChunkStreams] = {};         // stream si's last piece has been traced
    cudaEvent_t ev_rin[kChunkStreams] = {};        // stream si's input staging has been copied to the device
    cudaEvent_t ev_rout[kChunkStreams] = {};       // stream si's output scratch has been copied out
    // multi-view frames (tcrt_render_views): the call's camera table, copied in once per call; the pieces use the ray
    // batches' scratch, queue heads, counters and events above
    tcrt_camera* view_cams = nullptr;
    size_t view_cams_cap = 0;                      // cameras
    // sphere updates (tcrt_update_spheres): the upload's maps (slot_of, light_sph, levels, level_start) for the upload
    // numbered upd_serial, the input when it does not already live on this device, what the launches reduce (pinned copy
    // in h_upd_back), the spheres' boxes, and the grid's registration buffers — whose item list the scene then reads.
    // The call is synchronous: nothing else uses these while one runs.
    unsigned long long upd_serial = 0;
    int* upd_maps = nullptr;
    size_t upd_maps_cap = 0;                       // ints
    float4* upd_geom = nullptr;
    size_t upd_geom_cap = 0;
    unsigned char* upd_back = nullptr;
    size_t upd_back_cap = 0;
    unsigned char* h_upd_back = nullptr;
    size_t h_upd_back_cap = 0;
    float* upd_boxes = nullptr;
    size_t upd_boxes_cap = 0;                      // floats
    unsigned char* upd_grid = nullptr;
    size_t upd_grid_cap = 0;
    cudaEvent_t ev_u0 = nullptr, ev_u1 = nullptr;  // around the update's launches (render stream), or a material edit's
    // material edits (tcrt_update_materials): the object -> light map of the upload numbered mat_serial, and the records
    unsigned long long mat_serial = 0;
    int* mat_light_of = nullptr;
    size_t mat_light_of_cap = 0;                   // ints
    MaterialRecord* mat_rec = nullptr;
    size_t mat_rec_cap = 0;
    // plane updates (tcrt_update_planes): the finite-plane BVH's levels of the upload numbered pl_serial, its leaf boxes,
    // and the records
    unsigned long long pl_serial = 0;
    int* pl_levels = nullptr;
    size_t pl_levels_cap = 0;                      // ints
    float* pl_boxes = nullptr;
    size_t pl_boxes_cap = 0;                       // floats
    PlaneRecord* pl_rec = nullptr;
    size_t pl_rec_cap = 0;
};

struct TxtPipe;      // worker threads of the .txt writer and of the staged copy-out (defined with the writer)
struct TxtSink;

// Bounds on the colours a scene's paths form (DESIGN.md §4.1c), from its materials alone; dead_paths_prunable adds the
// launch's depth and NULL_COLOR.
struct DeadPathBound {
    bool finite = false;   // every colour, factor, intensity and texture colour is finite
    double local = 0.0;    // |local| of any level: every light's diffuse and specular terms, clamps ignored
    double leaf = 0.0;     // |tail| of a light hit or of a non-reflective hit (local)
    double obj = 0.0;      // largest |object colour| component, textures included
    double kref = 0.0;     // largest reflective factor
};

// ---- the per-launch scalars of the pruning structures (DeviceScene), from the bounds of what they hold -----------------
// Shared by the upload (plan_scene_blob) and by sphere updates (tcrt_update_spheres), which reduce the spheres' part of
// the bounds on the device and keep the planes' part from the upload.
struct SceneBounds {
    double sph_lo[3] = {1e300, 1e300, 1e300}, sph_hi[3] = {-1e300, -1e300, -1e300};   // boxes of the boxed spheres
    double pl_lo[3] = {1e300, 1e300, 1e300}, pl_hi[3] = {-1e300, -1e300, -1e300};     // finite-plane boxes, box clusters
    float rmin = INFINITY;                                                              // smallest radius in the sphere BVH
};

// bvh_rmin, bvh_c*, bvh_r2, bvh_cmax, clu_c*, clu_rbig, and grid_k2_max when the scene has a grid (grid_margin set)
void scene_scalars(const SceneBounds& b, bool sph_bvh, bool clusters, bool grid, DeviceScene& ds) {
    double blo[3], bhi[3];
    for (int k = 0; k < 3; k++) {
        blo[k] = std::min(b.sph_lo[k], b.pl_lo[k]);
        bhi[k] = std::max(b.sph_hi[k], b.pl_hi[k]);
    }
    ds.bvh_rmin = sph_bvh ? b.rmin * 0.999f : 1.f;
    ds.clu_cx = ds.clu_cy = ds.clu_cz = ds.clu_rbig = 0.f;
    ds.bvh_cx = ds.bvh_cy = ds.bvh_cz = ds.bvh_r2 = ds.bvh_cmax = 0.f;
    if (clusters) {
        double r1 = 0.0, cmax = 0.0;
        for (int k = 0; k < 3; k++) {
            r1 += 0.5 * (bhi[k] - blo[k]);
            cmax = std::max(cmax, std::max(fabs(blo[k]), fabs(bhi[k])));
        }
        ds.clu_cx = (float)(0.5 * (blo[0] + bhi[0]));
        ds.clu_cy = (float)(0.5 * (blo[1] + bhi[1]));
        ds.clu_cz = (float)(0.5 * (blo[2] + bhi[2]));
        ds.clu_rbig = (float)((r1 + cmax) * 1.001 + 1e-6);
    }
    if (ds.n_sph_bvh || ds.n_fin_bvh) {   // (a BVH that exists covers its prefix)
        double c[3], r2 = 0.0, cmax = 0.0;
        for (int k = 0; k < 3; k++) {
            if (!(blo[k] <= bhi[k])) blo[k] = bhi[k] = 0.0;
            c[k] = 0.5 * (blo[k] + bhi[k]);
            r2 += 0.25 * (bhi[k] - blo[k]) * (bhi[k] - blo[k]);
            cmax = std::max(cmax, std::max(fabs(blo[k]), fabs(bhi[k])));
        }
        ds.bvh_cx = (float)c[0]; ds.bvh_cy = (float)c[1]; ds.bvh_cz = (float)c[2];
        ds.bvh_r2 = (float)(r2 * 1.001 + 1e-6);
        ds.bvh_cmax = (float)(cmax * 1.001);
    }
    if (grid) {
        // the far-origin test without fatten()'s square root: m(k2) = (sqrt(rmin^2 + k2 E) - rmin) 1.001 + 1e-6 rmin grows
        // with k2, so m <= margin is a bound on k2 (solved in double, 0.1 % below: fewer rays on the grid is always sound)
        const double rmin = ds.bvh_rmin, t = ((double)ds.grid_margin - 1e-6 * rmin) / 1.001;
        const double k2 = t > 0.0 ? (t * t + 2.0 * t * rmin) / (double)TCRT_SPH_E : 0.0;
        ds.grid_k2_max = (float)(0.999 * k2);
    }
}

// The two light-table rows of a light at og: (position, intensity) (material colour, mask), what the light loop reads
// (RayTracer.cpp:540-563).  Shadow rays end at the light.  A cluster whose faces all lie on its hull ("shell": a room)
// cannot be crossed by a segment whose two ends are strictly inside the hull; whether the light is (with twice the
// kernel's per-ray margin) is a constant: bit c of the mask.  Needs ds.clu_* (scene_scalars).
void light_rows(const float* og, float intensity, const float* colour, const std::vector<TcrtBoxCluster>& clusters,
                const DeviceScene& ds, float4* rows) {
    unsigned inside_mask = 0u;
    for (int c = 0; c < (int)clusters.size() && c < 32; c++) {
        const TcrtBoxCluster& b = clusters[c];
        bool shell = true, inside = true;
        for (int f = 0; f < 6; f++)
            if (b.plane[f] >= 0 && b.c[f] != b.lo[f / 2] && b.c[f] != b.hi[f / 2]) shell = false;
        const double l1 = fabs((double)og[0] - ds.clu_cx) + fabs((double)og[1] - ds.clu_cy) +
                          fabs((double)og[2] - ds.clu_cz) + ds.clu_rbig;
        const double ml = 2.0 * 4e-6 * l1;   // 2 x TCRT_CLU_K x l1, see tcrt_render.cu clu_ray
        for (int k = 0; k < 3; k++)
            if (!((double)og[k] > (double)b.lo[k] + ml && (double)og[k] < (double)b.hi[k] - ml)) inside = false;
        if (shell && inside) inside_mask |= 1u << c;
    }
    rows[0] = make_float4(og[0], og[1], og[2], intensity);
    float4 lc = make_float4(colour[0], colour[1], colour[2], 0.f);
    memcpy(&lc.w, &inside_mask, 4);
    rows[1] = lc;
}

// The four blob rows of a box cluster (layout: tcrt_device.h)
void cluster_rows(const TcrtBoxCluster& b, float4* rows) {
    rows[0] = make_float4(b.lo[0], b.hi[0], b.lo[1], b.hi[1]);
    int present = 0;
    for (int f = 0; f < 6; f++) present |= (b.plane[f] >= 0) << f;
    float4 b1 = make_float4(b.lo[2], b.hi[2], 0.f, 0.f);
    memcpy(&b1.z, &present, 4);
    rows[1] = b1;
    rows[2] = make_float4(b.c[0], b.c[1], b.c[2], b.c[3]);
    rows[3] = make_float4(b.c[4], b.c[5], 0.f, 0.f);
}

// The six obj_normals rows of an object from its (facing, reverse) normals n8: per side the normal n1 the collision
// returns, n2 = normalize(n1) of Ray(point, normal) (Ray.h:21-25) and N = normalize(n2) of the specular term
// (RayTracer.cpp:565-566) — constants of the plane, evaluated with the reference's arithmetic (sqrtf, three divisions;
// this TU is built with -ffp-contract=off).  Shared by the upload and by plane updates, which must agree to the bit.
void normal_rows(const float* n8, float4* rows) {
    for (int side = 0; side < 2; side++) {
        float v[3] = {n8[4 * side], n8[4 * side + 1], n8[4 * side + 2]};
        for (int rep = 0; rep < 3; rep++) {
            rows[3 * side + rep] = make_float4(v[0], v[1], v[2], 0.f);
            volatile float len = sqrtf(v[0] * v[0] + v[1] * v[1] + v[2] * v[2]);   // vector3d.h:57-74
            v[0] = v[0] / len;
            v[1] = v[1] / len;
            v[2] = v[2] / len;
        }
    }
}

// What a sphere update needs of the upload: where each sphere lives in the blob, the planes' constants, the BVH's levels,
// the grid's registration arithmetic and the lights.  Plane updates (tcrt_update_planes) keep it current: it describes
// the resident scene, not only the upload.
struct UpdatePlan {
    int n_spheres = 0;
    std::vector<int> slot_of;            // sphere i (tcrt_scene order) -> its slot in the blob's sphere array (inverse of ps)
    int n_boxed = 0;                     // slots [0, n_boxed): the spheres the upload boxed into the bounds
    double ext_fixed = 1.0;              // max(1, |finite-plane origins|)
    double ext_sph = 0.0;                // max |sphere centre component|, of the upload or the last sphere update
    double ext_sph_box = 1.0;            // the ext the resident sphere boxes were built with
    double ext_fin_box = 1.0;            // the smallest ext a resident finite-plane box was built with
    SceneBounds bounds;                  // the spheres' part and the planes' part
    std::vector<int> levels, level_start;   // the sphere BVH's inner nodes, level by level from the root
    std::vector<TcrtBoxCluster> clusters;
    TcrtSphereGrid grid;                 // lo_d, cell_d, reg_margin_d, dims (no cells or items)
    size_t n_cells = 0;
    std::vector<float> light_og, light_col, light_int;   // 3, 3, 1 per light, current
    std::vector<int> light_sph;          // sphere index of each light sphere, in light order
    std::vector<int> light_of_sph;       // the light each of those is
    // planes (tcrt_update_planes): the blob's finite-plane rows by slot, each object's plane slot, the finite-plane BVH's
    // leaf boxes (6 per slot of its prefix) and inner levels, and the layout of the rows an update writes
    std::vector<float> fin_rows;         // 16 per finite-plane slot, as in the blob
    std::vector<int> fin_slot_of_obj, inf_slot_of_obj;   // object -> its finite / infinite plane slot, -1 for others
    std::vector<float> fin_boxes;
    std::vector<int> fin_levels, fin_level_start;
    size_t off_normals = 0, off_frame = 0;   // float4 offsets of obj_normals and inf_frame in the blob
};

// a box (lo xyz, hi xyz) into bounds lo, hi: its finite coordinates
void grow_into(double* lo, double* hi, const float* bx) {
    for (int k = 0; k < 3; k++) {
        if (std::isfinite(bx[k])) lo[k] = std::min(lo[k], (double)bx[k]);
        if (std::isfinite(bx[3 + k])) hi[k] = std::max(hi[k], (double)bx[3 + k]);
    }
}

// ext of the upload's boxes (plan_scene_blob), from its finite-plane part and its sphere part; update_ext in tcrt_update.cu
double scene_ext(double ext_fixed, double ext_sph) {
    const double ext = fmax(ext_fixed, ext_sph);
    return std::isfinite(ext) ? ext : 1e30;
}

// the level lists of a BVH's inner nodes from the root (tcrt_bvh.cpp: node 0), as the refit launch walks them
void bvh_levels(const std::vector<float4>& nodes, std::vector<int>& levels, std::vector<int>& level_start) {
    levels.clear();
    level_start.assign(1, 0);
    std::vector<int> level;
    if (!nodes.empty()) level.push_back(0);
    while (!level.empty()) {
        levels.insert(levels.end(), level.begin(), level.end());
        level_start.push_back((int)levels.size());
        std::vector<int> next;
        for (int node : level) {
            int ref[2];
            memcpy(ref, &nodes[4 * (size_t)node + 3], sizeof ref);   // (child0, child1, -, -)
            for (int r : ref)
                if (r >= 0) next.push_back(r);
        }
        level.swap(next);
    }
}

// What material edits (tcrt_update_materials, tcrt_update_textures) need of the last upload: a host copy of the scene's
// materials, with every edit merged in, and which light each object is.
struct MaterialShadow {
    std::vector<float> surface, material;   // obj_surface, obj_material
    std::vector<int> info;                  // obj_info: is_light and texture id are what the materials read
    std::vector<float> textures;
    std::vector<int> light_obj;
    std::vector<int> light_of;              // object index -> its light, -1 for the other objects
    int n_objects() const { return (int)(surface.size() / 4); }
    int n_textures() const { return (int)(textures.size() / 8); }
    // the parts of the scene dead_path_bound reads
    tcrt_scene view() const {
        tcrt_scene s{};
        s.n_objects = n_objects();
        s.n_lights = (int)light_obj.size();
        s.n_textures = n_textures();
        s.obj_surface = surface.data();
        s.obj_material = material.data();
        s.obj_info = info.data();
        s.light_obj = light_obj.data();
        s.textures = textures.data();
        return s;
    }
};

}  // namespace

static void destroy_copy_pipe(tcrt_ctx* ctx);

struct tcrt_ctx {
    std::vector<DeviceState> devs;
    TxtPipe* copy_pipe = nullptr;          // copy_out_staged's workers, started at the first pageable destination
    TxtSink* copy_sink = nullptr;
    std::string err;
    bool has_scene = false;
    bool has_frame = false;
    bool has_hits = false;       // a tcrt_hit_buffers call has completed (tcrt_device_hit_buffers)
    bool txt_prepared = false;
    int frame_x0 = 0, frame_x1 = 0, frame_h = 0;
    tcrt_camera cam{};           // passed by value with every launch
    // cached cost-balanced cut for the multi-device split (tcrt_balance_columns)
    std::vector<int> cut;
    tcrt_params cut_params{};
    bool cut_valid = false;
    // per-column cost estimate of the last tcrt_balance_columns (low resolution), for the same key
    std::vector<double> col_costs, row_costs;
    tcrt_params cost_params{};
    bool costs_valid = false;
    bool one_stream = false;               // developer builds: the chunk launches of a band on one stream, as before round 2
    unsigned long long cost_serial = 0;    // bumped by every new cost map
    char* host_text = nullptr;   // pinned staging for tcrt_write_txt
    size_t host_text_cap = 0;
    // frames in flight (tcrt_render_async): one per FrameRes set
    struct Pending {
        bool active = false;
        int x0 = 0, x1 = 0;
        tcrt_params params{};
        bool to_host = false;
        int launches = 0;
    } pend[2];
    // scene upload: pinned staging of the device blob, and the inputs it was built from (an unchanged scene
    // is not flattened, sorted and BVH-built again: tcrt_upload_scene then is a compare and one H2D copy)
    float4* scene_stage = nullptr;
    size_t scene_stage_cap = 0;     // float4s
    std::vector<unsigned char> scene_key;
    size_t scene_total_f4 = 0;
    int n_objects = 0;
    DeviceScene scene_ds{};
    size_t scene_off[9] = {};       // surface, material, normals, frame, tex, bvh_s, bvh_f, grid cells, grid items
    bool scene_bvh_s = false, scene_bvh_f = false, scene_grid = false;
    DeadPathBound scene_dead;
    UpdatePlan scene_upd;           // what tcrt_update_spheres needs of the last upload
    MaterialShadow scene_mat;       // what tcrt_update_materials and tcrt_update_textures need of it
    unsigned long long scene_serial = 0;   // bumped by every new blob (DeviceState::upd_serial, mat_serial)
    float4* upd_stage = nullptr;    // pinned: the input of tcrt_update_spheres, then the light rows it rewrites; the
                                    // packed records of a material edit
    size_t upd_stage_cap = 0;       // float4s
};

namespace {

thread_local std::string g_err = "";

int fail(tcrt_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    g_err = buf;
    return code;
}

#define CK(ctx, call)                                                                                        \
    do {                                                                                                     \
        cudaError_t e_ = (call);                                                                             \
        if (e_ != cudaSuccess)                                                                               \
            return fail(ctx, TCRT_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, \
                        __LINE__);                                                                           \
    } while (0)

template <typename T>
int ensure(tcrt_ctx* ctx, T*& p, size_t& cap, size_t need) {
    if (need <= cap && p) return TCRT_OK;
    if (p) CK(ctx, cudaFree(p));
    p = nullptr;
    cap = 0;
    CK(ctx, cudaMalloc((void**)&p, need * sizeof(T)));
    cap = need;
    return TCRT_OK;
}

void free_device(DeviceState& d) {
    if (d.dev < 0) return;
    cudaSetDevice(d.dev);
    if (d.stream) cudaStreamSynchronize(d.stream);
    for (auto& cs : d.chunk_stream)
        if (cs) cudaStreamSynchronize(cs);
    if (d.copy_stream) cudaStreamSynchronize(d.copy_stream);
    cudaFree(d.scene_mem);
    for (FrameRes& f : d.res) {
        cudaFree(f.frame);
        cudaFree(f.frame8);
        cudaFree(f.ctl);
        cudaFreeHost(f.h_counters);
        if (f.ev_start) cudaEventDestroy(f.ev_start);
        if (f.ev_k0) cudaEventDestroy(f.ev_k0);
        if (f.ev_k1) cudaEventDestroy(f.ev_k1);
        if (f.ev_c1) cudaEventDestroy(f.ev_c1);
        if (f.ev_done) cudaEventDestroy(f.ev_done);
        for (auto& e : f.ev_chunk)
            if (e) cudaEventDestroy(e);
    }
    if (d.ev_scene) cudaEventDestroy(d.ev_scene);
    cudaFree(d.text);
    cudaFree(d.offs);
    cudaFree(d.block_sums);
    cudaFree(d.flag);
    cudaFree(d.flush);
    cudaFree(d.row_order);
    cudaFree(d.col_cost);
    cudaFree(d.wave_mem);
    for (float* s : d.ss_scratch) cudaFree(s);
    cudaFree(d.hit_mem);
    cudaFree(d.pick_mem);
    cudaFree(d.hit_queue);
    cudaFree(d.ad_plain);
    cudaFree(d.ad_mask);
    cudaFree(d.ad_counts);
    cudaFree(d.ad_list);
    for (cudaEvent_t e : {d.ev_h0, d.ev_h1, d.ev_hc})
        if (e) cudaEventDestroy(e);
    for (int si = 0; si < kChunkStreams; si++) {
        cudaFree(d.ray_mem[si]);
        cudaFreeHost(d.ray_stage[si]);
        for (cudaEvent_t e : {d.ev_rk[si], d.ev_rin[si], d.ev_rout[si]})
            if (e) cudaEventDestroy(e);
    }
    cudaFree(d.ray_ctl);
    cudaFreeHost(d.h_ray);
    cudaFree(d.view_cams);
    cudaFree(d.upd_maps);
    cudaFree(d.upd_geom);
    cudaFree(d.upd_back);
    cudaFreeHost(d.h_upd_back);
    cudaFree(d.upd_boxes);
    cudaFree(d.upd_grid);
    cudaFree(d.mat_light_of);
    cudaFree(d.mat_rec);
    cudaFree(d.pl_levels);
    cudaFree(d.pl_boxes);
    cudaFree(d.pl_rec);
    for (cudaEvent_t e : {d.ev_u0, d.ev_u1})
        if (e) cudaEventDestroy(e);
    for (cudaEvent_t e : {d.ev_r0, d.ev_r1, d.ev_rc})
        if (e) cudaEventDestroy(e);
    cudaFreeHost(d.h_txt);
    cudaFreeHost(d.txt_stage);
    for (auto& e : d.ev_txt)
        if (e) cudaEventDestroy(e);
    for (auto& cs : d.chunk_stream)
        if (cs) cudaStreamDestroy(cs);
    if (d.copy_stream) cudaStreamDestroy(d.copy_stream);
    if (d.stream) cudaStreamDestroy(d.stream);
    d = DeviceState{};
}

// ---- conservative boxes for the BVH (all maths in double, then widened) ---------------------------
// A sphere hit point lies on the sphere; a finite-plane hit point P satisfies
// 0 <= (P-po).h <= h_dist and 0 <= (P-po).v <= v_dist (SceneFinitePlane.cpp:116-122) on the plane
// n.P = -dto.  h, v need not be orthogonal to each other or to n (three-corner ctor with skewed
// corners, or the axes ctor with a slanted normal), so the accepted region is the parallelogram cut
// out of the plane by the two slabs; its corners come from 2x2 solves in an in-plane basis.
void sphere_box(const float* g, double margin, float* box) {
    double r = sqrt(std::max(0.0, (double)g[3])) * (1.0 + 1e-6);
    for (int k = 0; k < 3; k++) {
        box[k] = (float)((double)g[k] - r - margin - 1e-6 * fabs((double)g[k]));
        box[3 + k] = (float)((double)g[k] + r + margin + 1e-6 * fabs((double)g[k]));
    }
}

void fin_box(const float* g, double margin, float* box) {
    const double n[3] = {g[0], g[1], g[2]}, h[3] = {g[4], g[5], g[6]}, v[3] = {g[8], g[9], g[10]};
    const double hd = g[7], vd = g[11], po[3] = {g[12], g[13], g[14]};
    auto unbounded = [&]() {
        for (int k = 0; k < 3; k++) { box[k] = -INFINITY; box[3 + k] = INFINITY; }
    };
    double nn = sqrt(n[0] * n[0] + n[1] * n[1] + n[2] * n[2]);
    if (!(nn > 1e-12) || !std::isfinite(nn) || !std::isfinite(hd) || !std::isfinite(vd)) return unbounded();
    double nu[3] = {n[0] / nn, n[1] / nn, n[2] / nn};
    // in-plane orthonormal basis e1, e2
    int m = fabs(nu[0]) < fabs(nu[1]) ? (fabs(nu[0]) < fabs(nu[2]) ? 0 : 2) : (fabs(nu[1]) < fabs(nu[2]) ? 1 : 2);
    double a[3] = {0, 0, 0};
    a[m] = 1.0;
    double e1[3] = {nu[1] * a[2] - nu[2] * a[1], nu[2] * a[0] - nu[0] * a[2], nu[0] * a[1] - nu[1] * a[0]};
    double l1 = sqrt(e1[0] * e1[0] + e1[1] * e1[1] + e1[2] * e1[2]);
    for (int k = 0; k < 3; k++) e1[k] /= l1;
    double e2[3] = {nu[1] * e1[2] - nu[2] * e1[1], nu[2] * e1[0] - nu[0] * e1[2], nu[0] * e1[1] - nu[1] * e1[0]};
    auto dot3 = [](const double* x, const double* y) { return x[0] * y[0] + x[1] * y[1] + x[2] * y[2]; };
    // constraints on q = (u, w), P - po = u e1 + w e2 :  0 <= a1.q <= hd,  0 <= a2.q <= vd
    double a1[2] = {dot3(h, e1), dot3(h, e2)}, a2[2] = {dot3(v, e1), dot3(v, e2)};
    double det = a1[0] * a2[1] - a1[1] * a2[0];
    double scale = sqrt((a1[0] * a1[0] + a1[1] * a1[1]) * (a2[0] * a2[0] + a2[1] * a2[1]));
    if (!(fabs(det) > 1e-6 * scale) || !(scale > 0)) return unbounded();
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    const double slack = 1e-5;   // the slab tests themselves are evaluated in float
    for (int ci = 0; ci < 4; ci++) {
        double x = (ci & 1) ? hd * (1 + slack) + slack : -slack * (1 + fabs(hd));
        double y = (ci & 2) ? vd * (1 + slack) + slack : -slack * (1 + fabs(vd));
        double u = (x * a2[1] - a1[1] * y) / det, w = (a1[0] * y - a2[0] * x) / det;
        for (int k = 0; k < 3; k++) {
            double c = po[k] + u * e1[k] + w * e2[k];
            lo[k] = std::min(lo[k], c);
            hi[k] = std::max(hi[k], c);
        }
    }
    for (int k = 0; k < 3; k++) {
        double pad = margin + 1e-5 * (fabs(lo[k]) + fabs(hi[k]) + (hi[k] - lo[k]));
        box[k] = (float)(lo[k] - pad);
        box[3 + k] = (float)(hi[k] + pad);
        if (!std::isfinite(box[k]) || !std::isfinite(box[3 + k])) { box[k] = -INFINITY; box[3 + k] = INFINITY; }
    }
}

// below these counts a linear sweep over shared memory is faster than a traversal
constexpr int kSphereBvhMin = 24;
constexpr int kFinBvhMin = 64;

bool valid_params(const tcrt_params* p) {
    return p && p->width > 0 && p->height > 0 && p->max_depth >= 0 &&
           (long long)p->width * (long long)p->height <= 0x7fffffffLL / 3;
}

}  // namespace

extern "C" {

int tcrt_abi_version(void) { return TCRT_ABI_VERSION; }

void tcrt_default_params(tcrt_params* p) {
    if (!p) return;
    p->width = 500;
    p->height = 504;
    p->max_depth = 50;
    p->shadows_on = 1;
    p->reflections_on = 1;
    p->null_color[0] = p->null_color[1] = p->null_color[2] = 0.75f;
    p->far_dist = 65535.0f;
}

int tcrt_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, TCRT_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    return n;
}

const char* tcrt_last_error(tcrt_ctx* ctx) { return ctx ? ctx->err.c_str() : g_err.c_str(); }

void* tcrt_alloc_host(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void tcrt_free_host(void* p) {
    if (p) cudaFreeHost(p);
}

int tcrt_create(tcrt_ctx** out, const int* device_ids, int n_devices) {
    if (!out || n_devices < 1 || n_devices > TCRT_MAX_DEVICES) return fail(nullptr, TCRT_ERR_INVALID, "bad arguments");
    *out = nullptr;
    int avail = tcrt_device_count();
    if (avail <= 0) return fail(nullptr, TCRT_ERR_NO_DEVICE, "no CUDA device available (%s)", g_err.c_str());
    tcrt_ctx* ctx = new tcrt_ctx();
#ifdef TCRT_DEV_KNOBS   // developer build only (A/B timing); the product never reads the environment
    ctx->one_stream = getenv("TCRT_ONE_STREAM") != nullptr;
#endif
    ctx->devs.resize(n_devices);
    for (int i = 0; i < n_devices; i++) {
        int dev = device_ids ? device_ids[i] : i;
        if (dev < 0 || dev >= avail) {
            tcrt_destroy(ctx);
            return fail(nullptr, TCRT_ERR_NO_DEVICE, "device %d out of range (have %d)", dev, avail);
        }
        DeviceState& d = ctx->devs[i];
        d.dev = dev;
        cudaError_t e = cudaSetDevice(dev);
        cudaDeviceProp prop;
        if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, dev);
        if (e == cudaSuccess && prop.major < 10) {
            tcrt_destroy(ctx);
            return fail(nullptr, TCRT_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", dev,
                        prop.major, prop.minor);
        }
        if (e == cudaSuccess) d.sm_count = prop.multiProcessorCount;
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking);
        for (auto& cs : d.chunk_stream)
            if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&cs, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&d.copy_stream, cudaStreamNonBlocking);
        for (FrameRes& f : d.res) {
            for (auto& ev : f.ev_chunk)
                if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f.ev_start, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaEventCreate(&f.ev_k0);
            if (e == cudaSuccess) e = cudaEventCreate(&f.ev_k1);
            if (e == cudaSuccess) e = cudaEventCreate(&f.ev_c1);
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&f.ev_done, cudaEventDisableTiming);
            if (e == cudaSuccess) e = cudaMalloc((void**)&f.ctl, 64 + kMaxChunks * sizeof(unsigned int));
            if (e == cudaSuccess) e = cudaHostAlloc((void**)&f.h_counters, 64, cudaHostAllocPortable);
        }
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&d.ev_scene, cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaMalloc((void**)&d.flag, 16);
        if (e == cudaSuccess) e = cudaMalloc((void**)&d.hit_queue, 16);
        if (e == cudaSuccess) e = cudaEventCreate(&d.ev_h0);
        if (e == cudaSuccess) e = cudaEventCreate(&d.ev_h1);
        if (e == cudaSuccess) e = cudaEventCreate(&d.ev_hc);
        if (e == cudaSuccess) e = cudaHostAlloc((void**)&d.h_txt, 64, cudaHostAllocPortable);
        if (e != cudaSuccess) {
            std::string msg = cudaGetErrorString(e);
            tcrt_destroy(ctx);
            return fail(nullptr, TCRT_ERR_CUDA, "device %d setup failed: %s", dev, msg.c_str());
        }
    }
    *out = ctx;
    return TCRT_OK;
}

void tcrt_destroy(tcrt_ctx* ctx) {
    if (!ctx) return;
    destroy_copy_pipe(ctx);
    for (auto& d : ctx->devs) free_device(d);
    if (ctx->host_text) cudaFreeHost(ctx->host_text);
    if (ctx->scene_stage) cudaFreeHost(ctx->scene_stage);
    if (ctx->upd_stage) cudaFreeHost(ctx->upd_stage);
    delete ctx;
}

// ---- scene upload -----------------------------------------------------------------------------
// What tcrt_upload_scene makes of a (validated) scene, on the host alone: the device blob and its description.
struct SceneBlob {
    std::vector<float4> host;
    DeviceScene ds{};
    size_t off[9] = {};          // surface, material, normals, frame, tex, bvh_s, bvh_f, grid cells, grid items
    bool grid = false, bvh_s = false, bvh_f = false;
    UpdatePlan upd;
    std::string err;
};
static int plan_scene_blob(const tcrt_scene* s, SceneBlob& out);
static int validate_scene(tcrt_ctx* ctx, const tcrt_scene* s);
static int build_scene_blob(tcrt_ctx* ctx, const tcrt_scene* s);
static int send_scene(tcrt_ctx* ctx, const tcrt_camera* cam);

static int validate_scene(tcrt_ctx* ctx, const tcrt_scene* s) {
    if (s->n_objects < 0 || s->n_spheres < 0 || s->n_fin_planes < 0 || s->n_inf_planes < 0 || s->n_lights < 0 ||
        s->n_textures < 0 || s->n_spheres + s->n_fin_planes + s->n_inf_planes != s->n_objects)
        return fail(ctx, TCRT_ERR_INVALID, "inconsistent scene counts");
    const int n = s->n_objects;
    for (int i = 0; i < s->n_spheres; i++)
        if (s->sphere_obj[i] < 0 || s->sphere_obj[i] >= n) return fail(ctx, TCRT_ERR_INVALID, "sphere_obj out of range");
    for (int i = 0; i < s->n_fin_planes; i++)
        if (s->fin_obj[i] < 0 || s->fin_obj[i] >= n) return fail(ctx, TCRT_ERR_INVALID, "fin_obj out of range");
    for (int i = 0; i < s->n_inf_planes; i++)
        if (s->inf_obj[i] < 0 || s->inf_obj[i] >= n) return fail(ctx, TCRT_ERR_INVALID, "inf_obj out of range");
    for (int i = 0; i < s->n_lights; i++)
        if (s->light_obj[i] < 0 || s->light_obj[i] >= n) return fail(ctx, TCRT_ERR_INVALID, "light_obj out of range");
    for (int i = 0; i < n; i++)
        if (s->obj_info[4 * i + 3] >= s->n_textures) return fail(ctx, TCRT_ERR_INVALID, "texture id out of range");
    return TCRT_OK;
}

// The grid kernel skips the shading of a level once every channel has met a zero object colour above it: that is exact
// only if every tail the reference forms (and k * tail) is finite, so that the zero turns it into +-0 and not into NaN
// (DESIGN.md §4.1c).  A bound in double: |dot| <= 1.001 for the unit vectors of the light loop (a cosine and the (V.R)
// of the specular term, whose 20th power is then <= 1.001^20), clamps ignored, leaf tails the NULL_COLOR, a light's
// colour (texture included) times its intensity, or a local colour; each stacked level adds its local colour to
// kref * obj * its child's.  The float arithmetic's relative error over a whole path stays below 1 %, far inside the
// margin to FLT_MAX that dead_paths_prunable keeps.
static DeadPathBound dead_path_bound(const tcrt_scene* s) {
    DeadPathBound b;
    const int n = s->n_objects;
    bool finite = true;
    auto fin = [&](float v) {
        finite = finite && std::isfinite(v);
        return fabs((double)v);
    };
    auto tex_max = [&](int t) {   // largest |component| of texture t's two colours
        double m = 0.0;
        for (int k = 0; k < 3; k++) m = std::max({m, fin(s->textures[8 * t + k]), fin(s->textures[8 * t + 4 + k])});
        return m;
    };
    double diffuse = 0.0, specular = 0.0, light_leaf = 0.0;
    for (int i = 0; i < n; i++) {
        double col = 0.0;
        for (int k = 0; k < 3; k++) col = std::max(col, fin(s->obj_surface[4 * i + k]));
        const int tex = s->obj_info[4 * i + 3];
        if (tex >= 0) col = std::max(col, tex_max(tex));
        b.obj = std::max(b.obj, col);
        diffuse = std::max(diffuse, fin(s->obj_surface[4 * i + 3]));
        specular = std::max(specular, fin(s->obj_material[4 * i]));
        b.kref = std::max(b.kref, fin(s->obj_material[4 * i + 1]));
        const double inten = fin(s->obj_material[4 * i + 2]);
        if (s->obj_info[4 * i + 2]) light_leaf = std::max(light_leaf, col * inten);
    }
    const double dot = 1.001, pw = pow(dot, 20.0);
    for (int l = 0; l < s->n_lights; l++) {
        const int lo = s->light_obj[l];
        double lc = 0.0;
        for (int k = 0; k < 3; k++) lc = std::max(lc, fabs((double)s->obj_surface[4 * lo + k]));
        // every factor taken as at least 1: then each partial product the light loop forms on the way — c * diffuse,
        // * intensity, * object colour (f * color * lc), and pw * specular — stays below its term as well, so no
        // intermediate can overflow to inf (and turn into NaN at a zero colour) while the bound stays small
        auto at_least_1 = [](double v) { return std::max(v, 1.0); };
        const double inten = fabs((double)s->obj_material[4 * lo + 2]);
        b.local += dot * at_least_1(diffuse) * at_least_1(inten) * at_least_1(b.obj) * at_least_1(lc) +
                   at_least_1(lc) * pw * at_least_1(specular);
    }
    b.leaf = std::max(light_leaf, b.local);
    b.finite = finite && std::isfinite(b.local);
    return b;
}

// Whether launches of `p` may skip dead levels: the scene's bound is finite and, over max_depth + 1 stacked levels below
// a leaf, every tail and every k * tail stays below 1e30 (FLT_MAX is 3.4e38).
static bool dead_paths_prunable(const DeadPathBound& b, const tcrt_params* p) {
    if (!b.finite) return false;
    double tail = 0.0;
    for (int k = 0; k < 3; k++) {
        if (!std::isfinite(p->null_color[k])) return false;
        tail = std::max(tail, fabs((double)p->null_color[k]));
    }
    tail = std::max(tail, b.leaf);
    const double limit = 1e30;
    for (int level = p->max_depth; level >= 0 && tail <= limit && b.kref * tail <= limit; level--)
        tail = b.local + b.kref * b.obj * tail;
    return tail <= limit && b.kref * tail <= limit;
}

int tcrt_plan_dead_paths(const tcrt_scene* s, const tcrt_params* p, int* prune) {
    if (!s || !p || !prune) return fail(nullptr, TCRT_ERR_INVALID, "null argument");
    if (!valid_params(p)) return fail(nullptr, TCRT_ERR_INVALID, "bad params");
    if (p->max_depth > TCRT_MAX_DEPTH) return fail(nullptr, TCRT_ERR_UNSUPPORTED, "max_depth too large");
    if (int rc = validate_scene(nullptr, s)) return rc;
    *prune = dead_paths_prunable(dead_path_bound(s), p) ? 1 : 0;
    return TCRT_OK;
}

int tcrt_upload_scene(tcrt_ctx* ctx, const tcrt_scene* s, const tcrt_camera* cam) {
    if (!ctx || !s || !cam) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (int rc = validate_scene(ctx, s)) return rc;
    const int n = s->n_objects;

    // ---- has this very scene been uploaded before?  (a caller that re-sends an unchanged scene every frame —
    // bench.py's e2e leg does — pays a compare and the H2D copy, not the sort + BVH/cluster build again)
    std::vector<unsigned char> key;
    {
        auto put = [&](const void* ptr, size_t bytes) {
            const unsigned char* b = static_cast<const unsigned char*>(ptr);
            key.insert(key.end(), b, b + bytes);
        };
        const int counts[6] = {s->n_objects, s->n_spheres, s->n_fin_planes, s->n_inf_planes, s->n_lights, s->n_textures};
        put(counts, sizeof counts);
        put(s->sphere_geom, sizeof(float) * 4 * s->n_spheres);
        put(s->sphere_obj, sizeof(int) * s->n_spheres);
        put(s->fin_geom, sizeof(float) * 16 * s->n_fin_planes);
        put(s->fin_obj, sizeof(int) * s->n_fin_planes);
        put(s->inf_geom, sizeof(float) * 16 * s->n_inf_planes);
        put(s->inf_obj, sizeof(int) * s->n_inf_planes);
        put(s->obj_surface, sizeof(float) * 4 * n);
        put(s->obj_material, sizeof(float) * 4 * n);
        put(s->obj_origin, sizeof(float) * 4 * n);
        put(s->obj_normals, sizeof(float) * 8 * n);
        put(s->obj_info, sizeof(int) * 4 * n);
        put(s->light_obj, sizeof(int) * s->n_lights);
        put(s->textures, sizeof(float) * 8 * s->n_textures);
    }
    const bool cached = ctx->has_scene && ctx->scene_stage != nullptr && key == ctx->scene_key;
    if (!cached) {
        int rc = build_scene_blob(ctx, s);
        if (rc) return rc;
        ctx->scene_key.swap(key);
    }
    return send_scene(ctx, cam);
}

// Flattened scene -> the device blob (sweep arrays, winner-only tables, BVH, box clusters) in ctx->scene_stage.
static int plan_scene_blob(const tcrt_scene* s, SceneBlob& out) {
    const int n = s->n_objects;
    auto is_light = [&](int obj) { return s->obj_info[4 * obj + 2] != 0; };
    // per type: non-light primitives first (shadow sweeps stop there), lights last
    auto order = [&](const int* objs, int cnt, std::vector<int>& perm, int& n_nl) {
        perm.clear();
        for (int i = 0; i < cnt; i++)
            if (!is_light(objs[i])) perm.push_back(i);
        n_nl = (int)perm.size();
        for (int i = 0; i < cnt; i++)
            if (is_light(objs[i])) perm.push_back(i);
    };
    std::vector<int> ps, pf, pi;
    DeviceScene ds{};
    ds.n_sph = s->n_spheres;
    ds.n_fin = s->n_fin_planes;
    ds.n_inf = s->n_inf_planes;
    ds.n_lights = s->n_lights;
    order(s->sphere_obj, s->n_spheres, ps, ds.n_sph_nl);
    order(s->fin_obj, s->n_fin_planes, pf, ds.n_fin_nl);
    order(s->inf_obj, s->n_inf_planes, pi, ds.n_inf_nl);

    // BVHs over the non-light primitives of a type when there are many; the covered prefix of the
    // type's array is re-ordered into leaf order.  `n_*_nl` keeps meaning "non-light" (the shadow
    // sweep's range); `n_*_bvh` <= n_*_nl is the BVH-covered prefix, the rest is swept linearly.
    std::vector<float4> bvh_s, bvh_f;
    TcrtSphereGrid grid;
    bool has_grid = false;
    int bvh_depth_s = 0, bvh_depth_f = 0;
    std::vector<TcrtBoxCluster> clusters;
    ds.n_fin_gen = ds.n_fin_nl;
    ds.n_arect = 0;
    ds.bvh_sph_root = ds.bvh_fin_root = 0;
    ds.n_sph_bvh = ds.n_fin_bvh = 0;
    UpdatePlan& upd = out.upd;
    SceneBounds& bounds = upd.bounds;
    {
        double ext = 1.0;
        for (int i = 0; i < s->n_fin_planes; i++)
            for (int k = 0; k < 3; k++) ext = std::max(ext, fabs((double)s->fin_geom[16 * i + 12 + k]));
        upd.ext_fixed = ext;
        for (int i = 0; i < s->n_spheres; i++)
            for (int k = 0; k < 3; k++) upd.ext_sph = std::max(upd.ext_sph, fabs((double)s->sphere_geom[4 * i + k]));
        ext = std::max(ext, upd.ext_sph);
        if (!std::isfinite(ext)) ext = 1e30;
        upd.ext_sph_box = upd.ext_fin_box = ext;
        const double margin = 1e-5 * ext;
        std::vector<float> boxes_s, boxes_f;
        std::vector<int> ord;
        auto grow_sph = [&](const float* bx) { grow_into(bounds.sph_lo, bounds.sph_hi, bx); };
        auto grow = [&](const float* bx) { grow_into(bounds.pl_lo, bounds.pl_hi, bx); };
        if (ds.n_sph_nl >= kSphereBvhMin) {
            // Tiny spheres would force a large per-ray fattening on everything (see `fatten`): the
            // (at most 16) spheres below half the median radius stay in the linear part.
            std::vector<float> rad(ds.n_sph_nl);
            for (int k = 0; k < ds.n_sph_nl; k++) rad[k] = sqrtf(std::max(0.f, s->sphere_geom[4 * ps[k] + 3]));
            std::vector<float> sorted(rad);
            std::sort(sorted.begin(), sorted.end());
            float r_cut = 0.5f * sorted[sorted.size() / 2];
            if (sorted.size() > 16 && sorted[16] < r_cut) r_cut = sorted[16];   // never more than 16 outside
            std::vector<int> in, out;
            for (int k = 0; k < ds.n_sph_nl; k++) (rad[k] >= r_cut && rad[k] > 0.f ? in : out).push_back(ps[k]);
            const int nb = (int)in.size();
            boxes_s.resize(6 * (size_t)nb);
            float rmin = INFINITY;
            for (int k = 0; k < nb; k++) {
                sphere_box(s->sphere_geom + 4 * in[k], margin, &boxes_s[6 * k]);
                grow_sph(&boxes_s[6 * k]);
                rmin = std::min(rmin, sqrtf(s->sphere_geom[4 * in[k] + 3]));
            }
            upd.n_boxed = nb;
            ds.bvh_sph_root = tcrt_build_bvh(boxes_s, nb, ord, bvh_s, &bvh_depth_s);
            std::vector<int> np;
            for (int k = 0; k < nb; k++) np.push_back(in[ord[k]]);
            np.insert(np.end(), out.begin(), out.end());
            np.insert(np.end(), ps.begin() + ds.n_sph_nl, ps.end());
            ps.swap(np);
            ds.n_sph_bvh = nb;
            bounds.rmin = rmin;
            // a uniform grid over the same spheres (leaf order), when they are even enough for one (tcrt_bvh.cpp)
            if (!bvh_s.empty()) {
                std::vector<float> leaf_boxes(6 * (size_t)nb);
                for (int k = 0; k < nb; k++) memcpy(&leaf_boxes[6 * (size_t)k], &boxes_s[6 * (size_t)ord[k]], 6 * sizeof(float));
                has_grid = tcrt_build_sphere_grid(leaf_boxes, nb, grid);
            }
            // The tree collapsed into one leaf (few spheres left after the exclusions, or SAH keeps
            // <= 8 coincident ones together): there are no nodes, the kernel variant without a sphere
            // BVH runs, and it stages and sweeps EVERY sphere — so none may count as BVH-covered.
            if (bvh_s.empty()) {
                ds.n_sph_bvh = 0;
                ds.bvh_sph_root = 0;
                bvh_depth_s = 0;
            }
        }
        if (ds.n_fin_nl >= kFinBvhMin) {
            boxes_f.resize(6 * (size_t)ds.n_fin_nl);
            for (int k = 0; k < ds.n_fin_nl; k++) {
                fin_box(s->fin_geom + 16 * pf[k], margin, &boxes_f[6 * k]);
                grow(&boxes_f[6 * k]);
            }
            ds.bvh_fin_root = tcrt_build_bvh(boxes_f, ds.n_fin_nl, ord, bvh_f, &bvh_depth_f);
            std::vector<int> np(pf);
            for (int k = 0; k < ds.n_fin_nl; k++) np[k] = pf[ord[k]];
            pf.swap(np);
            ds.n_fin_bvh = ds.n_fin_nl;
            if (!bvh_f.empty()) {   // the leaf boxes by slot, for plane updates
                upd.fin_boxes.resize(6 * (size_t)ds.n_fin_nl);
                for (int k = 0; k < ds.n_fin_nl; k++)
                    memcpy(&upd.fin_boxes[6 * (size_t)k], &boxes_f[6 * (size_t)ord[k]], 6 * sizeof(float));
            }
        }
        // Axis-aligned finite planes (every makeSceneBox face) are swept through box clusters instead
        // of one by one (tcrt_cluster.cpp); with a finite-plane BVH the BVH covers them.
        if (bvh_f.empty() && ds.n_fin_nl > 0) {
            std::vector<int> cand(pf.begin(), pf.begin() + ds.n_fin_nl), is_arect;
            tcrt_build_box_clusters(s->fin_geom, cand, is_arect, clusters);
            // a handful of rectangles is swept one by one: the cluster code would only cost
            // instruction-cache space (the reference's SCENE 2 has four finite planes)
            int n_rect = 0;
            for (int a : is_arect) n_rect += a != 0;
            if (n_rect < 6) clusters.clear();
            if (!clusters.empty()) {
                std::vector<int> np, new_pos(ds.n_fin_nl, -1);
                for (int k = 0; k < ds.n_fin_nl; k++)
                    if (!is_arect[k]) { new_pos[k] = (int)np.size(); np.push_back(pf[k]); }
                ds.n_fin_gen = (int)np.size();
                for (int k = 0; k < ds.n_fin_nl; k++)
                    if (is_arect[k]) { new_pos[k] = (int)np.size(); np.push_back(pf[k]); }
                ds.n_arect = (int)np.size() - ds.n_fin_gen;
                np.insert(np.end(), pf.begin() + ds.n_fin_nl, pf.end());
                pf.swap(np);
                for (auto& c : clusters) {
                    for (int f = 0; f < 6; f++)
                        if (c.plane[f] >= 0) c.plane[f] = new_pos[c.plane[f]];   // -> slot in the finite-plane array
                    grow(c.lo);   // lo[3], hi[3] are contiguous: a 6-float box
                }
            }
        }
    }

    ds.fin_off = ds.n_sph;
    ds.inf_off = ds.fin_off + 4 * ds.n_fin;
    ds.light_off = ds.inf_off + ds.n_inf;
    ds.n_clu = (int)clusters.size();
    ds.clu_off = ds.light_off + 2 * ds.n_lights;
    ds.cslot_off = ds.clu_off + 4 * ds.n_clu;
    ds.idx_off = ds.cslot_off + (6 * ds.n_clu + 3) / 4;
    const int n_prims = ds.n_sph + ds.n_fin + ds.n_inf;
    ds.blob_f4 = ds.idx_off + (n_prims + 3) / 4;
    if (std::max(bvh_depth_s, bvh_depth_f) + 2 > TCRT_BVH_STACK)   // cannot happen below ~2^40 primitives (tcrt_bvh.cpp)
        return out.err = "BVH depth " + std::to_string(std::max(bvh_depth_s, bvh_depth_f)) + " exceeds the traversal stack", TCRT_ERR_UNSUPPORTED;
    ds.stage_off = ds.n_sph_bvh;   // BVH leaves read their spheres through L1
    if ((size_t)(ds.blob_f4 - ds.stage_off) * sizeof(float4) > tcrt_render_max_smem())
        return out.err = "scene needs " + std::to_string((size_t)(ds.blob_f4 - ds.stage_off) * sizeof(float4)) +
                         " B of shared memory per CTA (limit " + std::to_string(tcrt_render_max_smem()) + ")",
               TCRT_ERR_UNSUPPORTED;

    const size_t off_surface = (size_t)ds.blob_f4;
    const size_t off_material = off_surface + n;
    const size_t off_normals = off_material + n;
    const size_t off_frame = off_normals + 6 * (size_t)n;
    const size_t off_tex = off_frame + 3 * (size_t)ds.n_inf;
    const size_t off_bvh_s = off_tex + 2 * (size_t)s->n_textures;
    const size_t off_bvh_f = off_bvh_s + bvh_s.size();
    // the grid serves the kernels without finite-plane structures (FM 0 / 3); elsewhere the sphere BVH alone
    has_grid = has_grid && !bvh_s.empty() && bvh_f.empty() && clusters.empty();
    if (has_grid) {
        for (int k = 0; k < 3; k++) {
            ds.grid_lo[k] = grid.lo[k];
            ds.grid_cell[k] = grid.cell[k];
            ds.grid_hi[k] = grid.lo[k] + grid.cell[k] * (float)grid.dims[k];
            ds.grid_inv_cell[k] = 1.0f / grid.cell[k];
            ds.grid_dims[k] = grid.dims[k];
        }
        ds.grid_margin = grid.reg_margin;
    }
    scene_scalars(bounds, !bvh_s.empty(), !clusters.empty(), has_grid, ds);
    const size_t off_grid_cells = off_bvh_f + bvh_f.size();
    const size_t n_grid_cells = has_grid ? grid.cell_start.size() - 1 : 0;
    const size_t off_grid_items = off_grid_cells + 2 * n_grid_cells;
    const size_t total_f4 = off_grid_items + (has_grid ? (grid.items.size() + 3) / 4 : 0) + 1;
    std::vector<float4> host(total_f4, make_float4(0.f, 0.f, 0.f, 0.f));
    auto f4 = [](const float* p) { return make_float4(p[0], p[1], p[2], p[3]); };
    int* idx = reinterpret_cast<int*>(&host[ds.idx_off]);
    for (int k = 0; k < ds.n_sph; k++) {
        host[k] = f4(s->sphere_geom + 4 * ps[k]);
        idx[k] = s->sphere_obj[ps[k]];
    }
    for (int k = 0; k < ds.n_fin; k++) {
        for (int j = 0; j < 4; j++) host[ds.fin_off + 4 * k + j] = f4(s->fin_geom + 16 * pf[k] + 4 * j);
        idx[ds.n_sph + k] = s->fin_obj[pf[k]];
    }
    for (int k = 0; k < ds.n_inf; k++) {
        host[ds.inf_off + k] = f4(s->inf_geom + 16 * pi[k]);
        for (int j = 0; j < 3; j++) host[off_frame + 3 * k + j] = f4(s->inf_geom + 16 * pi[k] + 4 * (j + 1));
        idx[ds.n_sph + ds.n_fin + k] = s->inf_obj[pi[k]];
    }
    {
        int* cslot = reinterpret_cast<int*>(&host[ds.cslot_off]);
        for (int c = 0; c < ds.n_clu; c++) {
            const TcrtBoxCluster& b = clusters[c];
            cluster_rows(b, &host[ds.clu_off + 4 * c]);
            for (int f = 0; f < 6; f++) cslot[6 * c + f] = b.plane[f];
        }
    }
    for (int l = 0; l < ds.n_lights; l++) {
        const int lo = s->light_obj[l];
        light_rows(s->obj_origin + 4 * lo, s->obj_material[4 * lo + 2], s->obj_surface + 4 * lo, clusters, ds,
                   &host[ds.light_off + 2 * l]);
    }
    for (int i = 0; i < n; i++) {
        host[off_surface + i] = f4(s->obj_surface + 4 * i);
        float4 m = f4(s->obj_material + 4 * i);
        int flags = (s->obj_info[4 * i + 3] + 1) & 0x7fffffff;
        if (is_light(i)) flags |= (int)0x80000000u;
        memcpy(&m.w, &flags, sizeof(float));   // bit pattern, read back with __float_as_int
        host[off_material + i] = m;
        normal_rows(s->obj_normals + 8 * (size_t)i, &host[off_normals + 6 * (size_t)i]);
    }
    for (int t = 0; t < s->n_textures; t++) {
        host[off_tex + 2 * t] = f4(s->textures + 8 * t);
        host[off_tex + 2 * t + 1] = f4(s->textures + 8 * t + 4);
    }
    std::copy(bvh_s.begin(), bvh_s.end(), host.begin() + off_bvh_s);
    std::copy(bvh_f.begin(), bvh_f.end(), host.begin() + off_bvh_f);
    if (has_grid) {
        // cell record: the first sphere's geometry next to the cell's count, so a one-sphere cell is one round of loads
        for (size_t c = 0; c < n_grid_cells; c++) {
            const int j0 = grid.cell_start[c], cnt = grid.cell_start[c + 1] - j0;
            int4 meta = make_int4(cnt > 0 ? cnt - 1 : 0, cnt > 0 ? grid.items[j0] : 0, j0 + 1, 0);
            // spheres sit at the front of the blob; an empty cell gets a sphere whose discriminant is negative for every ray
            host[off_grid_cells + 2 * c] = cnt > 0 ? host[grid.items[j0]] : make_float4(0.f, 0.f, 0.f, -1e30f);
            memcpy(&host[off_grid_cells + 2 * c + 1], &meta, sizeof(meta));
        }
        memcpy(&host[off_grid_items], grid.items.data(), grid.items.size() * sizeof(int));
    }

    // what a sphere update needs (tcrt_update_spheres)
    upd.n_spheres = ds.n_sph;
    upd.slot_of.assign(ds.n_sph, 0);
    for (int k = 0; k < ds.n_sph; k++) upd.slot_of[ps[k]] = k;
    bvh_levels(bvh_s, upd.levels, upd.level_start);
    bvh_levels(bvh_f, upd.fin_levels, upd.fin_level_start);
    upd.fin_rows.resize(16 * (size_t)ds.n_fin);
    for (int k = 0; k < ds.n_fin; k++) memcpy(&upd.fin_rows[16 * (size_t)k], s->fin_geom + 16 * (size_t)pf[k], 16 * sizeof(float));
    upd.fin_slot_of_obj.assign(n, -1);
    upd.inf_slot_of_obj.assign(n, -1);
    for (int k = 0; k < ds.n_fin; k++) upd.fin_slot_of_obj[s->fin_obj[pf[k]]] = k;
    for (int k = 0; k < ds.n_inf; k++) upd.inf_slot_of_obj[s->inf_obj[pi[k]]] = k;
    upd.off_normals = off_normals;
    upd.off_frame = off_frame;
    upd.clusters = clusters;
    if (has_grid) {
        upd.grid = grid;
        upd.grid.cell_start.clear();
        upd.grid.items.clear();
        upd.n_cells = n_grid_cells;
    }
    std::vector<int> sph_of_obj(n, -1);   // the sphere whose centre an object's origin is (the last, should several share one)
    for (int i = 0; i < s->n_spheres; i++) sph_of_obj[s->sphere_obj[i]] = i;
    for (int l = 0; l < ds.n_lights; l++) {
        const int lo = s->light_obj[l];
        for (int k = 0; k < 3; k++) {
            upd.light_og.push_back(s->obj_origin[4 * lo + k]);
            upd.light_col.push_back(s->obj_surface[4 * lo + k]);
        }
        upd.light_int.push_back(s->obj_material[4 * lo + 2]);
        if (sph_of_obj[lo] >= 0) {
            upd.light_sph.push_back(sph_of_obj[lo]);
            upd.light_of_sph.push_back(l);
        }
    }

    out.ds = ds;
    out.off[0] = off_surface;
    out.off[1] = off_material;
    out.off[2] = off_normals;
    out.off[3] = off_frame;
    out.off[4] = off_tex;
    out.off[5] = off_bvh_s;
    out.off[6] = off_bvh_f;
    out.off[7] = off_grid_cells;
    out.off[8] = off_grid_items;
    out.grid = has_grid;
    out.bvh_s = !bvh_s.empty();
    out.bvh_f = !bvh_f.empty();
    out.host.swap(host);
    return TCRT_OK;
}

static int build_scene_blob(tcrt_ctx* ctx, const tcrt_scene* s) {
    SceneBlob b;
    const int rc = plan_scene_blob(s, b);
    if (rc) return fail(ctx, rc, "%s", b.err.c_str());
    const size_t total_f4 = b.host.size();
    // into the pinned staging buffer (once every device has finished reading the previous scene out of it)
    for (auto& d : ctx->devs) {
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaEventSynchronize(d.ev_scene));
    }
    if (total_f4 > ctx->scene_stage_cap) {
        if (ctx->scene_stage) cudaFreeHost(ctx->scene_stage);
        ctx->scene_stage = nullptr;
        ctx->scene_stage_cap = 0;
        CK(ctx, cudaHostAlloc((void**)&ctx->scene_stage, total_f4 * sizeof(float4), cudaHostAllocPortable));
        ctx->scene_stage_cap = total_f4;
    }
    memcpy(ctx->scene_stage, b.host.data(), total_f4 * sizeof(float4));
    ctx->scene_total_f4 = total_f4;
    ctx->n_objects = s->n_objects;
    ctx->scene_ds = b.ds;
    for (int k = 0; k < 9; k++) ctx->scene_off[k] = b.off[k];
    ctx->scene_grid = b.grid;
    ctx->scene_bvh_s = b.bvh_s;
    ctx->scene_bvh_f = b.bvh_f;
    ctx->scene_dead = dead_path_bound(s);
    ctx->scene_upd = std::move(b.upd);
    {
        const int n = s->n_objects;
        MaterialShadow& m = ctx->scene_mat;
        m.surface.assign(s->obj_surface, s->obj_surface + 4 * (size_t)n);
        m.material.assign(s->obj_material, s->obj_material + 4 * (size_t)n);
        m.info.assign(s->obj_info, s->obj_info + 4 * (size_t)n);
        m.textures.assign(s->textures, s->textures + 8 * (size_t)s->n_textures);
        m.light_obj.assign(s->light_obj, s->light_obj + s->n_lights);
        m.light_of.assign(n, -1);
        for (int l = 0; l < s->n_lights; l++) m.light_of[s->light_obj[l]] = l;
    }
    ctx->scene_serial++;
    return TCRT_OK;
}

// Staged blob -> every device of the ctx, asynchronously on the render stream (frames queued earlier still see
// the previous scene, frames queued later the new one); the camera travels with every launch.
static int send_scene(tcrt_ctx* ctx, const tcrt_camera* cam) {
    const size_t total_f4 = ctx->scene_total_f4;
    for (auto& d : ctx->devs) {
        CK(ctx, cudaSetDevice(d.dev));
        int rc = ensure(ctx, d.scene_mem, d.scene_cap_f4, total_f4);
        if (rc) return rc;
        CK(ctx, cudaMemcpyAsync(d.scene_mem, ctx->scene_stage, total_f4 * sizeof(float4), cudaMemcpyHostToDevice, d.stream));
        CK(ctx, cudaEventRecord(d.ev_scene, d.stream));
        d.ds = ctx->scene_ds;
        d.ds.blob = d.scene_mem;
        d.ds.obj_surface = d.scene_mem + ctx->scene_off[0];
        d.ds.obj_material = d.scene_mem + ctx->scene_off[1];
        d.ds.obj_normals = d.scene_mem + ctx->scene_off[2];
        d.ds.inf_frame = d.scene_mem + ctx->scene_off[3];
        d.ds.textures = d.scene_mem + ctx->scene_off[4];
        d.ds.obj_info = nullptr;
        d.ds.bvh_sph = ctx->scene_bvh_s ? d.scene_mem + ctx->scene_off[5] : nullptr;
        d.ds.bvh_fin = ctx->scene_bvh_f ? d.scene_mem + ctx->scene_off[6] : nullptr;
        d.ds.grid_cells = ctx->scene_grid ? d.scene_mem + ctx->scene_off[7] : nullptr;
        d.ds.grid_items = ctx->scene_grid ? reinterpret_cast<const int*>(d.scene_mem + ctx->scene_off[8]) : nullptr;
    }
    ctx->cam = *cam;
    ctx->cut_valid = false;
    ctx->costs_valid = false;
    ctx->has_scene = true;
    ctx->has_frame = false;
    ctx->txt_prepared = false;
    return TCRT_OK;
}

// ---- render -------------------------------------------------------------------------------------
int tcrt_rebalance_columns(const int* bounds, const double* ms, int n_bands, int width, int* new_bounds) {
    if (!bounds || !ms || !new_bounds || n_bands < 1 || width < 0) return TCRT_ERR_INVALID;
    if (bounds[0] != 0 || bounds[n_bands] != width) return TCRT_ERR_INVALID;
    std::vector<double> cost((size_t)std::max(width, 1), 0.0);
    for (int b = 0; b < n_bands; b++) {
        const int w = bounds[b + 1] - bounds[b];
        if (w < 0 || !(ms[b] >= 0.0)) return TCRT_ERR_INVALID;
        for (int x = bounds[b]; x < bounds[b + 1]; x++) cost[x] = ms[b] / w;
    }
    if (width == 0) {
        for (int b = 0; b <= n_bands; b++) new_bounds[b] = 0;
        return TCRT_OK;
    }
    return tcrt_bands_from_costs(cost.data(), width, width, n_bands, new_bounds);
}

static int launch_band(tcrt_ctx* ctx, DeviceState& d, const tcrt_params* p, int cx0, int cx1, float* out, unsigned int* col_cost,
                       int* launches, cudaStream_t stream = nullptr, unsigned int* queue = nullptr);
static int ensure_row_order(tcrt_ctx* ctx, DeviceState& d, const tcrt_params* p, int cx0, int cx1, bool pre_pass, const int** out);

// Samples per axis of a supersampled frame (tcrt_render_columns_ss).  At 8 the widest column chunk of a 7680x4320 frame
// needs 2.2 GB of sample scratch per render stream (DESIGN.md §4.3).
constexpr int kMaxSS = 8;

// The column chunks of a device band [f.x0, f.x1) -> f.n_chunks, f.chunk_x.  px_per_col: pixels traced per column of the
// band (ss*ss*height for a supersampled frame).  Unchunked: one launch.  Chunked (a host destination, or a supersampled
// frame): up to kMaxChunks column chunks.  Chunk k of a band that goes to host memory is copied back on the copy stream
// while the next chunks render (the output is x-major: a chunk is one contiguous slice).  The chunks are separate launches
// on kChunkStreams streams, round robin: a launch ends in a tail of half-empty SMs (its deepest paths: 0.13-0.25 ms per
// launch measured), and with the next chunks' launches already queued on the other streams their CTAs move in as this
// one's retire.
static void plan_chunks(FrameRes& f, long long px_per_col, bool chunked) {
    const int w = f.x1 - f.x0;
    int n_chunks = 1;
    if (chunked) {
        // 256 K pixels (3 MB) or more per chunk: a 1080p frame is 7 chunks (0.56 ms end to end; 3 chunks 0.61 ms,
        // 15 chunks 0.57 ms), larger frames kMaxChunks
        const long long chunk_px = 256 * 1024;
        n_chunks = (int)std::min<long long>(std::min<long long>(kMaxChunks, w), std::max<long long>(1, w * px_per_col / chunk_px));
    }
    // chunk boundaries on tile boundaries, so that every chunk of a tileable band is tileable.  With the full
    // number of chunks the first and the last ones are narrow: the copies start after the first chunk's kernel
    // and the frame ends with the last chunk's copy, neither of which anything hides.
    static const int kChunkWeight[kMaxChunks + 1] = {0, 1, 2, 4, 8, 12, 16, 20, 24, 28, 32, 36, 40, 42, 44, 45, 46};
    for (int j = 0; j <= n_chunks; j++) {
        int c = n_chunks == kMaxChunks ? (int)((long long)w * kChunkWeight[j] / kChunkWeight[kMaxChunks])
                                       : (int)((long long)w * j / n_chunks);
        if (j < n_chunks && w % TCRT_TILE_W == 0) c -= c % TCRT_TILE_W;
        f.chunk_x[j] = f.x0 + c;
    }
    f.n_chunks = n_chunks;
}

// One frame = submit (everything is queued on the devices' streams, nothing waits) + finish (waits for this
// frame's events only, reads its timings and ray counters).  `set` picks which of the two FrameRes sets of
// every device the frame lives in.
// copies: how a band gets to the host.  kCopyDirect: cudaMemcpyAsync of every chunk into host_band (pinned memory: truly
// asynchronous).  kCopyStaged: chunked launches and their events only — the caller moves the chunks out afterwards
// (copy_out_staged: pageable destinations).  Ignored without host_band.
enum { kCopyDirect = 0, kCopyStaged = 1 };
// What crosses the bus: the float32 frame, or (tcrt_render_rgb8) each chunk quantised by one more launch on its stream into
// the device's byte buffer.  The float frame stays the "last render" either way.
enum FrameFormat { kFloat32 = 0, kRGB8 = 1 };
static size_t bytes_per_px(FrameFormat fmt) { return fmt == kRGB8 ? 3 : 3 * sizeof(float); }
static const char* frame_src(const FrameRes& f, FrameFormat fmt) {
    return fmt == kRGB8 ? reinterpret_cast<const char*>(f.frame8) : reinterpret_cast<const char*>(f.frame);
}
// ss > 1: a supersampled frame (tcrt_render_columns_ss).  Chunk k of output columns [c0, c1) is one render launch over
// sample columns [ss*c0, ss*c1) of the sample frame (ss*width x ss*height) into the scratch buffer of its stream, then one
// resolve launch on that stream into the band's frame (and, for RGB8, its byte buffer).  The caller has checked ss.
static int render_submit(tcrt_ctx* ctx, const tcrt_params* p, int x0, int x1, void* host_band, int set, int copies = kCopyDirect,
                         FrameFormat fmt = kFloat32, int ss = 1) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null ctx");
    if (!valid_params(p)) return fail(ctx, TCRT_ERR_INVALID, "bad params");
    if (x0 < 0 || x1 > p->width || x0 >= x1) return fail(ctx, TCRT_ERR_INVALID, "bad column range [%d,%d)", x0, x1);
    if (p->max_depth > TCRT_MAX_DEPTH)
        return fail(ctx, TCRT_ERR_UNSUPPORTED, "max_depth %d > TCRT_MAX_DEPTH %d", p->max_depth, TCRT_MAX_DEPTH);
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    if (ctx->pend[set].active)
        return fail(ctx, TCRT_ERR_INVALID, "a frame submitted with tcrt_render_async is still pending in this slot: tcrt_wait first");
    const int nd = (int)ctx->devs.size();
    const int cols = x1 - x0;
    if (set == ctx->devs[0].cur) {
        ctx->has_frame = false;
        ctx->txt_prepared = false;
    }
    int launches = 0;
    // one contiguous band of columns per device (x-major storage makes a band one slice)
    // (cost-balanced over the whole image when it is rendered whole; equal widths for a sub-range)
    std::vector<int> cut(nd + 1);
    for (int i = 0; i <= nd; i++) cut[i] = x0 + (int)((long long)cols * i / nd);
    if (nd > 1 && x0 == 0 && x1 == p->width) {
        const bool same = ctx->cut_valid && (int)ctx->cut.size() == nd + 1 && ctx->cut_params.width == p->width &&
                          ctx->cut_params.height == p->height && ctx->cut_params.max_depth == p->max_depth &&
                          ctx->cut_params.shadows_on == p->shadows_on && ctx->cut_params.reflections_on == p->reflections_on;
        if (!same) {
            ctx->cut.assign(nd + 1, 0);
            int rc = tcrt_balance_columns(ctx, p, nd, ctx->cut.data());
            if (rc) return rc;
            ctx->cut_params = *p;
            ctx->cut_valid = true;
        }
        cut = ctx->cut;
    }
    const int prev_cur = ctx->devs[0].cur;
    const bool super = ss > 1;
    tcrt_params sp = *p;                // the frame the render launches trace: for a supersampled frame, its sample frame
    sp.width = ss * p->width;
    sp.height = ss * p->height;
    const long long spc = (long long)ss * sp.height;     // pixels traced per output column
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        d.cur = set;
        d.fr().x0 = cut[i];
        d.fr().x1 = cut[i + 1];
        d.fr().height = p->height;
        if (d.fr().x1 <= d.fr().x0) continue;
        plan_chunks(d.fr(), spc, host_band != nullptr || super);
        // the render kernels index the pixels of a launch with ints (3 floats each)
        for (int k = 0; super && k < d.fr().n_chunks; k++)
            if ((long long)(d.fr().chunk_x[k + 1] - d.fr().chunk_x[k]) * spc > 0x7fffffffLL / 3) {
                for (auto& dd : ctx->devs) dd.cur = prev_cur;
                return fail(ctx, TCRT_ERR_UNSUPPORTED, "%d x %d at %d x %d samples: a column chunk of the sample frame exceeds "
                            "the kernels' index range", p->width, p->height, ss, ss);
            }
    }
    auto submit_all = [&]() -> int {
        for (int i = 0; i < nd; i++) {
            DeviceState& d = ctx->devs[i];
            if (d.fr().x1 <= d.fr().x0) continue;
            CK(ctx, cudaSetDevice(d.dev));
            const size_t n_floats = (size_t)(d.fr().x1 - d.fr().x0) * p->height * 3;
            int rc = ensure(ctx, d.fr().frame, d.fr().frame_cap, n_floats);
            if (rc) return rc;
            if (fmt == kRGB8 && host_band) {
                rc = ensure(ctx, d.fr().frame8, d.fr().frame8_cap, n_floats);
                if (rc) return rc;
            }
            CK(ctx, cudaMemsetAsync(d.fr().ctl, 0, 64, d.stream));
            const int n_chunks = d.fr().n_chunks;
            const int* chunk_x = d.fr().chunk_x;
            const bool two_streams = n_chunks > 1 && !ctx->one_stream;   // (several streams)
            if (super) {       // sample scratch for the widest chunk, on every stream the chunks use
                int widest = 0;
                for (int k = 0; k < n_chunks; k++) widest = std::max(widest, chunk_x[k + 1] - chunk_x[k]);
                const size_t need = (size_t)widest * spc * 3;
                const int n_bufs = two_streams ? std::min(kChunkStreams, n_chunks) : 1;
                for (int si = 0; si < n_bufs; si++)     // a buffer about to be replaced may still serve the other frame set
                    if (need > d.ss_scratch_cap[si]) {
                        CK(ctx, cudaDeviceSynchronize());
                        break;
                    }
                for (int si = 0; si < n_bufs; si++) {
                    rc = ensure(ctx, d.ss_scratch[si], d.ss_scratch_cap[si], need);
                    if (rc) return rc;
                }
            }
            if (two_streams) {
                // everything the launches on the second stream read must be in place: queue heads, counters, row order
                CK(ctx, cudaMemsetAsync(d.fr().ctl + 64, 0, kMaxChunks * sizeof(unsigned int), d.stream));
                const int* unused = nullptr;
                rc = ensure_row_order(ctx, d, &sp, ss * chunk_x[0], ss * chunk_x[1], false, &unused);
                if (rc) return rc;
                CK(ctx, cudaEventRecord(d.fr().ev_start, d.stream));
                for (auto& cs : d.chunk_stream) CK(ctx, cudaStreamWaitEvent(cs, d.fr().ev_start, 0));
            }
            CK(ctx, cudaEventRecord(d.fr().ev_k0, d.stream));
            int last_on[kChunkStreams];
            for (int& l : last_on) l = -1;
            for (int k = 0; k < n_chunks; k++) {
                const int cx0 = chunk_x[k], cx1 = chunk_x[k + 1];
                if (cx1 <= cx0) continue;
                const size_t off = (size_t)(cx0 - d.fr().x0) * p->height * 3;     // channels into the band
                const size_t cnt = (size_t)(cx1 - cx0) * p->height * 3;
                cudaStream_t ks = d.stream;
                const int si = two_streams ? k % kChunkStreams : 0;
                float* out = super ? d.ss_scratch[si] : d.fr().frame + off;
                if (two_streams) {
                    if (si > 0) ks = d.chunk_stream[si - 1];
                    last_on[si] = k;
                    rc = launch_band(ctx, d, &sp, ss * cx0, ss * cx1, out, nullptr, &launches, ks,
                                     reinterpret_cast<unsigned int*>(d.fr().ctl + 64) + k);
                } else {
                    if (k > 0) CK(ctx, cudaMemsetAsync(d.fr().ctl, 0, 4, d.stream));   // queue head only; ray counters accumulate
                    rc = launch_band(ctx, d, &sp, ss * cx0, ss * cx1, out, nullptr, &launches);
                }
                if (rc) return rc;
                if (super) {
                    CK(ctx, tcrt_launch_resolve_ss(out, cx1 - cx0, p->height, ss, d.fr().frame + off,
                                                   fmt == kRGB8 && host_band ? d.fr().frame8 + off : nullptr, ks));
                    launches++;
                }
                if (host_band || super) {
                    if (host_band && fmt == kRGB8 && !super) {
                        CK(ctx, tcrt_launch_quantize8(d.fr().frame + off, cnt / 3, d.fr().frame8 + off, ks));
                        launches++;
                    }
                    CK(ctx, cudaEventRecord(d.fr().ev_chunk[k], ks));
                    if (host_band && copies == kCopyDirect) {
                        const size_t bpc = bytes_per_px(fmt) / 3;                      // bytes per channel
                        CK(ctx, cudaStreamWaitEvent(d.copy_stream, d.fr().ev_chunk[k], 0));
                        CK(ctx, cudaMemcpyAsync(static_cast<char*>(host_band) + ((size_t)(d.fr().x0 - x0) * p->height * 3 + off) * bpc,
                                                frame_src(d.fr(), fmt) + off * bpc, cnt * bpc, cudaMemcpyDeviceToHost, d.copy_stream));
                    }
                }
            }
            for (int si = 1; si < kChunkStreams; si++)      // the frame ends on d.stream
                if (last_on[si] >= 0) CK(ctx, cudaStreamWaitEvent(d.stream, d.fr().ev_chunk[last_on[si]], 0));
            CK(ctx, cudaEventRecord(d.fr().ev_k1, d.stream));
            CK(ctx, cudaMemcpyAsync(d.fr().h_counters, d.fr().ctl, 32, cudaMemcpyDeviceToHost, d.stream));
            CK(ctx, cudaEventRecord(d.fr().ev_done, d.stream));
            if (host_band && copies == kCopyDirect) CK(ctx, cudaEventRecord(d.fr().ev_c1, d.copy_stream));
        }
        return TCRT_OK;
    };
    const int rc = submit_all();
    if (rc) {
        for (auto& d : ctx->devs) d.cur = prev_cur;
        return rc;
    }
    tcrt_ctx::Pending& pd = ctx->pend[set];
    pd.active = true;
    pd.x0 = x0;
    pd.x1 = x1;
    pd.params = *p;
    pd.to_host = host_band != nullptr && copies == kCopyDirect;
    pd.launches = launches;
    return TCRT_OK;
}

static int render_finish(tcrt_ctx* ctx, int set, tcrt_stats* stats) {
    tcrt_ctx::Pending& pd = ctx->pend[set];
    if (!pd.active) return fail(ctx, TCRT_ERR_INVALID, "no frame pending in slot %d", set);
    const int nd = (int)ctx->devs.size();
    const tcrt_params* p = &pd.params;
    for (auto& d : ctx->devs) d.cur = set;
    pd.active = false;
    if (stats) memset(stats, 0, sizeof(*stats));
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        if (stats) {
            stats->col_begin[i] = d.fr().x0;
            stats->col_end[i] = d.fr().x1;
        }
        if (d.fr().x1 <= d.fr().x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        // this frame's events only: a later frame may already be queued behind it on the same streams
        CK(ctx, cudaEventSynchronize(d.fr().ev_done));
        if (pd.to_host) CK(ctx, cudaEventSynchronize(d.fr().ev_c1));
        if (stats) {
            float ms = 0.f;
            CK(ctx, cudaEventElapsedTime(&ms, d.fr().ev_k0, d.fr().ev_k1));
            stats->render_ms[i] = ms;
            if (pd.to_host) CK(ctx, cudaEventElapsedTime(&ms, d.fr().ev_k1, d.fr().ev_c1));
            stats->d2h_ms[i] = pd.to_host ? std::max(ms, 0.f) : 0.0;   // copy time not hidden behind the render
            stats->rays_primary[i] = d.fr().h_counters[1];
            stats->rays_shadow[i] = d.fr().h_counters[2];
            stats->rays_reflect[i] = d.fr().h_counters[3];
        }
    }
    if (stats) {
        stats->n_devices = nd;
        stats->gpu_launches = (unsigned long long)pd.launches;
    }
    // feedback: the next frame with these params is cut by this frame's measured band times
    if (nd > 1 && pd.x0 == 0 && pd.x1 == p->width && ctx->cut_valid && (int)ctx->cut.size() == nd + 1) {
        std::vector<double> ms(nd, 0.0);
        std::vector<int> next(nd + 1, 0), used(nd + 1, 0);
        bool ok = true;
        for (int i = 0; i < nd; i++) {
            DeviceState& d = ctx->devs[i];
            float t = 0.f;
            if (d.fr().x1 > d.fr().x0) ok = ok && cudaEventElapsedTime(&t, d.fr().ev_k0, d.fr().ev_k1) == cudaSuccess;
            ms[i] = t;
            used[i] = d.fr().x0;
        }
        used[nd] = p->width;     // the cut THIS frame was rendered with (a later frame may already have moved ctx->cut)
        if (ok && tcrt_rebalance_columns(used.data(), ms.data(), nd, p->width, next.data()) == TCRT_OK) ctx->cut = next;
    }
    ctx->has_frame = true;
    ctx->txt_prepared = false;
    ctx->frame_x0 = pd.x0;
    ctx->frame_x1 = pd.x1;
    ctx->frame_h = p->height;
    return TCRT_OK;
}

static int copy_out_staged(tcrt_ctx* ctx, const tcrt_params* p, int x0, void* host_band, FrameFormat fmt);

static int render_impl(tcrt_ctx* ctx, const tcrt_params* p, int x0, int x1, void* host_band, tcrt_stats* stats,
                       FrameFormat fmt = kFloat32, int ss = 1) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null ctx");
    const int set = ctx->devs[0].cur;
    // A pageable destination (a plain malloc'd / std::vector / numpy buffer): cudaMemcpyAsync would block the calling
    // thread chunk by chunk and move the data at the driver's staging rate (measured 13-14 GB/s).  Instead every chunk goes
    // to pinned staging at bus speed and worker threads copy it on (copy_out_staged).
    bool staged = false;
    if (host_band && valid_params(p) && x0 >= 0 && x1 <= p->width && (long long)(x1 - x0) * p->height >= 512 * 1024) {
        cudaPointerAttributes at{};
        if (cudaPointerGetAttributes(&at, host_band) != cudaSuccess) {
            cudaGetLastError();
            staged = true;
        } else {
            staged = at.type == cudaMemoryTypeUnregistered;
        }
    }
    int rc = render_submit(ctx, p, x0, x1, host_band, set, staged ? kCopyStaged : kCopyDirect, fmt, ss);
    if (rc) return rc;
    if (staged) {
        rc = copy_out_staged(ctx, p, x0, host_band, fmt);
        if (rc) {
            render_finish(ctx, set, nullptr);
            return rc;
        }
    }
    return render_finish(ctx, set, stats);
}

// The launch of columns [cx0, cx1) of the frame `p` into `out`, with queue head `queue` (nullptr: the frame set's) and the
// frame set's ray counters; no row order, no cost map.
static RenderLaunch band_launch(tcrt_ctx* ctx, DeviceState& d, const tcrt_params* p, int cx0, int cx1, float* out,
                                unsigned int* queue) {
    RenderLaunch rl{};
    rl.scene = d.ds;
    rl.cam = ctx->cam;
    rl.width = p->width;
    rl.height = p->height;
    rl.x0 = cx0;
    rl.x1 = cx1;
    rl.max_depth = p->max_depth;
    rl.shadows_on = p->shadows_on;
    rl.reflections_on = p->reflections_on;
    rl.null_r = p->null_color[0];
    rl.null_g = p->null_color[1];
    rl.null_b = p->null_color[2];
    rl.far_dist = p->far_dist;
    rl.prune_dead = dead_paths_prunable(ctx->scene_dead, p) ? 1 : 0;
    rl.n_objects = ctx->n_objects;
    rl.out = out;
    rl.queue = queue ? queue : reinterpret_cast<unsigned int*>(d.fr().ctl);
    rl.counters = reinterpret_cast<unsigned long long*>(d.fr().ctl + 8);
    return rl;
}

// Columns [cx0, cx1) of the frame `p` into out[(cx1-cx0)*p->height*3] (a slice of the band's frame buffer, or the sample
// scratch of a supersampled frame, whose `p` is then the sample frame).  The caller has sized out and zeroed the queue head.
static int launch_band(tcrt_ctx* ctx, DeviceState& d, const tcrt_params* p, int cx0, int cx1, float* out, unsigned int* col_cost,
                       int* launches, cudaStream_t stream, unsigned int* queue) {
    if (!stream) stream = d.stream;
    RenderLaunch rl = band_launch(ctx, d, p, cx0, cx1, out, queue);
    rl.col_cost = col_cost;
    int rc_ro = ensure_row_order(ctx, d, p, cx0, cx1, col_cost != nullptr, &rl.row_order);
    if (rc_ro) return rc_ro;
    // scratch of the wavefront path (large frames of sphere-BVH scenes): ray queues and per-path state of one chunk
    const size_t wave_need = tcrt_wave_mem_needed(rl);
    if (wave_need > d.wave_bytes) {
        if (d.wave_mem) CK(ctx, cudaFree(d.wave_mem));
        d.wave_mem = nullptr;
        d.wave_bytes = 0;
        CK(ctx, cudaMalloc(&d.wave_mem, wave_need));
        d.wave_bytes = wave_need;
    }
    CK(ctx, tcrt_launch_render(rl, d.sm_count, stream, launches, d.wave_mem, d.wave_bytes));
    return TCRT_OK;
}

// Longest-processing-time-first: with a cost map for this (scene, camera, params) — i.e. after
// tcrt_balance_columns — the queue runs row by row, the expensive rows first, so the tail of the
// launch is made of cheap pixels (sky, floor) instead of the deepest reflection paths, whose
// bounces are sequential and would otherwise drain on an almost empty GPU.  *out = the device's row order for a
// launch over columns [cx0, cx1) (uploaded on d.stream when it is not there yet), or nullptr.
static int ensure_row_order(tcrt_ctx* ctx, DeviceState& d, const tcrt_params* p, int cx0, int cx1, bool pre_pass, const int** out) {
    *out = nullptr;
    const tcrt_params& cp = ctx->cost_params;
    if (ctx->costs_valid && !pre_pass && p->height > 1 && cp.width == p->width && cp.height == p->height &&
        cp.max_depth == p->max_depth && cp.shadows_on == p->shadows_on && cp.reflections_on == p->reflections_on) {
        // rows, or 8-row tile rows when the launch is tiled (same rule as tcrt_launch_render)
        const bool tiled = (cx1 - cx0) % TCRT_TILE_W == 0 && p->height % TCRT_TILE_H == 0;
        const int unit = tiled ? TCRT_TILE_H : 1;
        const int key_h = tiled ? -p->height : p->height;
        if (d.row_order_serial != ctx->cost_serial || d.row_order_h != key_h || !d.row_order) {
            const int n = p->height / unit, nl = (int)ctx->row_costs.size();
            std::vector<int> order(n);
            for (int i = 0; i < n; i++) order[i] = i;
            auto cost_of = [&](int r) {
                double c = 0.0;
                for (int k = 0; k < unit; k++)
                    c += ctx->row_costs[std::min(nl - 1, (int)((long long)(r * unit + k) * nl / p->height))];
                return c;
            };
            std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return cost_of(a) > cost_of(b); });
            int rc = ensure(ctx, d.row_order, d.row_order_cap, (size_t)n);
            if (rc) return rc;
            CK(ctx, cudaMemcpyAsync(d.row_order, order.data(), sizeof(int) * n, cudaMemcpyHostToDevice, d.stream));
            d.row_order_serial = ctx->cost_serial;
            d.row_order_h = key_h;
        }
        *out = d.row_order;
    }
    return TCRT_OK;
}

int tcrt_render(tcrt_ctx* ctx, const tcrt_params* p, float* host_rgb, tcrt_stats* stats) {
    if (!host_rgb) return fail(ctx, TCRT_ERR_INVALID, "null output buffer");
    if (!p) return fail(ctx, TCRT_ERR_INVALID, "null params");
    return render_impl(ctx, p, 0, p->width, host_rgb, stats);
}
int tcrt_render_columns(tcrt_ctx* ctx, const tcrt_params* p, int x0, int x1, float* host_rgb_band, tcrt_stats* stats) {
    if (!host_rgb_band) return fail(ctx, TCRT_ERR_INVALID, "null output buffer");
    return render_impl(ctx, p, x0, x1, host_rgb_band, stats);
}
int tcrt_render_device(tcrt_ctx* ctx, const tcrt_params* p, int x0, int x1, tcrt_stats* stats) {
    return render_impl(ctx, p, x0, x1, nullptr, stats);
}

static int render_async_impl(tcrt_ctx* ctx, const tcrt_params* p, int x0, int x1, void* host_band, int* ticket, FrameFormat fmt,
                             int ss = 1) {
    if (!ctx || !ticket) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    // the set that is not pending; with none pending, the one the last frame did not use (its band may still be wanted)
    int set = ctx->pend[0].active ? 1 : (ctx->pend[1].active ? 0 : 1 - ctx->devs[0].cur);
    if (ctx->pend[set].active) return fail(ctx, TCRT_ERR_INVALID, "two frames are already in flight: tcrt_wait for one first");
    const int keep = ctx->devs[0].cur;
    int rc = render_submit(ctx, p, x0, x1, host_band, set, kCopyDirect, fmt, ss);
    if (rc) return rc;
    // the "last frame" of the synchronous calls (tcrt_download, the writers) stays what it was until tcrt_wait
    for (auto& d : ctx->devs) d.cur = keep;
    *ticket = set;
    return TCRT_OK;
}

int tcrt_render_async(tcrt_ctx* ctx, const tcrt_params* p, int x0, int x1, float* host_rgb_band, int* ticket) {
    return render_async_impl(ctx, p, x0, x1, host_rgb_band, ticket, kFloat32);
}

// ---- 8-bit frames: the same calls, each column chunk quantised on the device before it crosses the bus --------------
int tcrt_render_rgb8(tcrt_ctx* ctx, const tcrt_params* p, unsigned char* host_rgb8, tcrt_stats* stats) {
    if (!host_rgb8) return fail(ctx, TCRT_ERR_INVALID, "null output buffer");
    if (!p) return fail(ctx, TCRT_ERR_INVALID, "null params");
    return render_impl(ctx, p, 0, p->width, host_rgb8, stats, kRGB8);
}
int tcrt_render_columns_rgb8(tcrt_ctx* ctx, const tcrt_params* p, int x0, int x1, unsigned char* host_rgb8_band,
                             tcrt_stats* stats) {
    if (!host_rgb8_band) return fail(ctx, TCRT_ERR_INVALID, "null output buffer");
    return render_impl(ctx, p, x0, x1, host_rgb8_band, stats, kRGB8);
}
int tcrt_render_async_rgb8(tcrt_ctx* ctx, const tcrt_params* p, int x0, int x1, unsigned char* host_rgb8_band, int* ticket) {
    if (!host_rgb8_band) return fail(ctx, TCRT_ERR_INVALID, "null output buffer");
    return render_async_impl(ctx, p, x0, x1, host_rgb8_band, ticket, kRGB8);
}

// ---- supersampled frames: ss x ss samples of the reference's frame at (ss*width, ss*height) per pixel, box-filtered ------
// ss = 1 is the plain frame through the plain path.
static int check_ss(tcrt_ctx* ctx, const tcrt_params* p, int ss) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null ctx");
    if (ss < 1) return fail(ctx, TCRT_ERR_INVALID, "samples per axis %d < 1", ss);
    if (ss > kMaxSS) return fail(ctx, TCRT_ERR_UNSUPPORTED, "samples per axis %d > %d", ss, kMaxSS);
    // the kernels map sample column x to (float)x / (float)(ss*width): exact up to 2^24
    if (p && ((long long)ss * p->width > (1LL << 24) || (long long)ss * p->height > (1LL << 24)))
        return fail(ctx, TCRT_ERR_UNSUPPORTED, "sample frame %lld x %lld: above 2^24 columns or rows",
                    (long long)ss * p->width, (long long)ss * p->height);
    return TCRT_OK;
}
int tcrt_render_columns_ss(tcrt_ctx* ctx, const tcrt_params* p, int ss, int x0, int x1, float* host_rgb_band, tcrt_stats* stats) {
    const int rc = check_ss(ctx, p, ss);
    return rc ? rc : render_impl(ctx, p, x0, x1, host_rgb_band, stats, kFloat32, ss);
}
int tcrt_render_columns_ss_rgb8(tcrt_ctx* ctx, const tcrt_params* p, int ss, int x0, int x1, unsigned char* host_rgb8_band,
                                tcrt_stats* stats) {
    if (!host_rgb8_band) return fail(ctx, TCRT_ERR_INVALID, "null output buffer");
    const int rc = check_ss(ctx, p, ss);
    return rc ? rc : render_impl(ctx, p, x0, x1, host_rgb8_band, stats, kRGB8, ss);
}
int tcrt_render_async_ss(tcrt_ctx* ctx, const tcrt_params* p, int ss, int x0, int x1, float* host_rgb_band, int* ticket) {
    const int rc = check_ss(ctx, p, ss);
    return rc ? rc : render_async_impl(ctx, p, x0, x1, host_rgb_band, ticket, kFloat32, ss);
}
int tcrt_render_async_ss_rgb8(tcrt_ctx* ctx, const tcrt_params* p, int ss, int x0, int x1, unsigned char* host_rgb8_band,
                              int* ticket) {
    if (!host_rgb8_band) return fail(ctx, TCRT_ERR_INVALID, "null output buffer");
    const int rc = check_ss(ctx, p, ss);
    return rc ? rc : render_async_impl(ctx, p, x0, x1, host_rgb8_band, ticket, kRGB8, ss);
}

int tcrt_wait(tcrt_ctx* ctx, int ticket, tcrt_stats* stats) {
    if (!ctx || ticket < 0 || ticket > 1) return fail(ctx, TCRT_ERR_INVALID, "bad ticket");
    return render_finish(ctx, ticket, stats);
}

int tcrt_download(tcrt_ctx* ctx, float* host_band) {
    if (!ctx || !host_band) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (!ctx->has_frame) return fail(ctx, TCRT_ERR_NO_FRAME, "nothing rendered yet");
    // a large pageable destination: through pinned staging and the ctx's copy workers, like tcrt_render (render_impl)
    if ((long long)(ctx->frame_x1 - ctx->frame_x0) * ctx->frame_h >= 512 * 1024) {
        cudaPointerAttributes at{};
        bool pageable;
        if (cudaPointerGetAttributes(&at, host_band) != cudaSuccess) {
            cudaGetLastError();
            pageable = true;
        } else {
            pageable = at.type == cudaMemoryTypeUnregistered;
        }
        if (pageable) {
            tcrt_params p{};
            p.height = ctx->frame_h;
            return copy_out_staged(ctx, &p, ctx->frame_x0, host_band, kFloat32);
        }
    }
    for (auto& d : ctx->devs) {
        if (d.fr().x1 <= d.fr().x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        const size_t n_floats = (size_t)(d.fr().x1 - d.fr().x0) * d.fr().height * 3;
        float* dst = host_band + (size_t)(d.fr().x0 - ctx->frame_x0) * d.fr().height * 3;
        CK(ctx, cudaMemcpyAsync(dst, d.fr().frame, n_floats * sizeof(float), cudaMemcpyDeviceToHost, d.stream));
    }
    for (auto& d : ctx->devs) {
        if (d.fr().x1 <= d.fr().x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));
    }
    return TCRT_OK;
}

int tcrt_bands_from_costs(const double* costs, int n_costs, int width, int n_bands, int* bounds) {
    if (!costs || !bounds || n_costs < 1 || width < 0 || n_bands < 1) return TCRT_ERR_INVALID;
    double total = 0.0;
    for (int i = 0; i < n_costs; i++) {
        if (!(costs[i] >= 0.0)) return TCRT_ERR_INVALID;
        total += costs[i];
    }
    bounds[0] = 0;
    bounds[n_bands] = width;
    int j = 0;              // current cost group
    double before = 0.0;    // cost of groups [0, j)
    for (int k = 1; k < n_bands; k++) {
        int b;
        if (!(total > 0.0)) {
            b = (int)((long long)width * k / n_bands);
        } else {
            const double target = total * k / n_bands;
            while (j < n_costs - 1 && before + costs[j] < target) before += costs[j++];
            const double frac = costs[j] > 0.0 ? std::min(1.0, std::max(0.0, (target - before) / costs[j])) : 0.0;
            b = (int)floor(((double)j + frac) * width / n_costs + 0.5);
        }
        bounds[k] = std::min(width, std::max(bounds[k - 1], b));
    }
    // The kernel hands out 4-column x 8-row tiles when a band's width is a multiple of 4
    // (tcrt_render.cu): interior cuts move to the nearest multiple of 4 — two columns of imbalance
    // at most — unless the bands are only a few columns wide.
    if (width % TCRT_TILE_W == 0 && width >= 4 * TCRT_TILE_W * n_bands)
        for (int k = 1; k < n_bands; k++)
            bounds[k] = std::min(width, std::max(bounds[k - 1], ((bounds[k] + TCRT_TILE_W / 2) / TCRT_TILE_W) * TCRT_TILE_W));
    return TCRT_OK;
}

int tcrt_balance_columns(tcrt_ctx* ctx, const tcrt_params* p, int n_bands, int* bounds) {
    if (!ctx || !bounds || n_bands < 1) return fail(ctx, TCRT_ERR_INVALID, "bad arguments");
    if (!valid_params(p)) return fail(ctx, TCRT_ERR_INVALID, "bad params");
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    if (p->max_depth > TCRT_MAX_DEPTH) return fail(ctx, TCRT_ERR_UNSUPPORTED, "max_depth too large");
    if (n_bands == 1) {
        bounds[0] = 0;
        bounds[1] = p->width;
        return TCRT_OK;
    }
    // low-resolution copy of the frame: same camera percentages (Camera.cpp:71-84 maps x/W, z/H)
    tcrt_params lp = *p;
    lp.width = std::min(p->width, 256);
    lp.height = std::max(1, std::min(p->height, (int)((long long)p->height * lp.width / std::max(1, p->width))));
    DeviceState& d = ctx->devs[0];
    CK(ctx, cudaSetDevice(d.dev));
    // the pre-pass borrows the device's frame buffer and band bookkeeping
    ctx->has_frame = false;
    ctx->txt_prepared = false;
    d.fr().x0 = 0;
    d.fr().x1 = lp.width;
    d.fr().height = lp.height;
    const size_t n_cost = (size_t)lp.width + lp.height;    // per column, then per row
    int rc = ensure(ctx, d.col_cost, d.col_cost_cap, n_cost);
    if (rc) return rc;
    unsigned int* col_cost = d.col_cost;
    std::vector<unsigned int> h(n_cost);
    int launches = 0;
    cudaError_t e = cudaMemsetAsync(col_cost, 0, sizeof(unsigned int) * n_cost, d.stream);
    if (e == cudaSuccess) rc = ensure(ctx, d.fr().frame, d.fr().frame_cap, (size_t)lp.width * lp.height * 3);
    if (e == cudaSuccess && rc == TCRT_OK) e = cudaMemsetAsync(d.fr().ctl, 0, 64, d.stream);
    if (e == cudaSuccess && rc == TCRT_OK) rc = launch_band(ctx, d, &lp, 0, lp.width, d.fr().frame, col_cost, &launches);
    if (e == cudaSuccess && rc == TCRT_OK)
        e = cudaMemcpyAsync(h.data(), col_cost, sizeof(unsigned int) * n_cost, cudaMemcpyDeviceToHost, d.stream);
    if (e == cudaSuccess && rc == TCRT_OK) e = cudaStreamSynchronize(d.stream);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(ctx, TCRT_ERR_CUDA, "balance pre-pass failed: %s", cudaGetErrorString(e));
    std::vector<double> costs(h.begin(), h.begin() + lp.width);
    ctx->col_costs = costs;
    ctx->row_costs.assign(h.begin() + lp.width, h.end());
    ctx->cost_params = *p;
    ctx->costs_valid = true;
    ctx->cost_serial++;
    if (tcrt_bands_from_costs(costs.data(), lp.width, p->width, n_bands, bounds) != TCRT_OK)
        return fail(ctx, TCRT_ERR_INVALID, "bands_from_costs failed");
    return TCRT_OK;
}

int tcrt_device_frame(tcrt_ctx* ctx, int slot, void** dev_ptr, size_t* n_floats) {
    if (!ctx || slot < 0 || slot >= (int)ctx->devs.size() || !dev_ptr || !n_floats)
        return fail(ctx, TCRT_ERR_INVALID, "bad argument");
    if (!ctx->has_frame) return fail(ctx, TCRT_ERR_NO_FRAME, "nothing rendered yet");
    DeviceState& d = ctx->devs[slot];
    *dev_ptr = d.fr().frame;
    *n_floats = (size_t)(d.fr().x1 - d.fr().x0) * d.fr().height * 3;
    return TCRT_OK;
}

int tcrt_flush_l2(tcrt_ctx* ctx) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null ctx");
    const size_t bytes = (size_t)256 << 20;   // > the 126 MB L2
    for (auto& d : ctx->devs) {
        CK(ctx, cudaSetDevice(d.dev));
        if (!d.flush) {
            CK(ctx, cudaMalloc(&d.flush, bytes));
            d.flush_bytes = bytes;
        }
        CK(ctx, tcrt_launch_l2_flush(d.flush, d.flush_bytes, d.stream));
    }
    for (auto& d : ctx->devs) {
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));
    }
    return TCRT_OK;
}

int tcrt_fp32_peak(tcrt_ctx* ctx, double* unfused, double* fma, double* ms_each) {
    if (!ctx || !unfused || !fma) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    DeviceState& d = ctx->devs[0];
    CK(ctx, cudaSetDevice(d.dev));
    const int grid = d.sm_count * 8;      // 8 CTAs x 8 warps = the full 64 warps per SM
    const int iters = 1 << 16;
    double res[2] = {0, 0}, ms_out[2] = {0, 0};
    for (int mode = 0; mode < 2; mode++) {
        float best = 1e30f;
        for (int rep = 0; rep < 4; rep++) {   // first rep warms up
            CK(ctx, cudaEventRecord(d.fr().ev_k0, d.stream));
            CK(ctx, tcrt_launch_fp32_peak(mode == 1, reinterpret_cast<float*>(d.flag), grid, iters, d.stream));
            CK(ctx, cudaEventRecord(d.fr().ev_k1, d.stream));
            CK(ctx, cudaStreamSynchronize(d.stream));
            float ms = 0.f;
            CK(ctx, cudaEventElapsedTime(&ms, d.fr().ev_k0, d.fr().ev_k1));
            if (rep > 0 && ms < best) best = ms;
        }
        const double lane_inst = (double)grid * 256.0 * (double)iters * 8.0 * (mode == 1 ? 1.0 : 2.0);
        res[mode] = lane_inst / (best * 1e-3) / 1e12;
        ms_out[mode] = best;
    }
    *unfused = res[0];
    *fma = res[1];
    if (ms_each) { ms_each[0] = ms_out[0]; ms_each[1] = ms_out[1]; }
    return TCRT_OK;
}

static void fill_structures(const DeviceScene& ds, bool grid, bool bvh_s, bool bvh_f, int info[8]) {
    info[0] = bvh_s ? ds.n_sph_bvh : 0;                                                  // spheres in the sphere BVH
    info[1] = grid ? ds.grid_dims[0] * ds.grid_dims[1] * ds.grid_dims[2] : 0;            // cells of the sphere grid
    info[2] = bvh_f ? ds.n_fin_bvh : 0;                                                  // finite planes in their BVH
    info[3] = ds.n_clu;                                                                  // box clusters
    info[4] = ds.n_arect;                                                                // rectangles owned by clusters
    info[5] = ds.n_sph - (bvh_s ? ds.n_sph_bvh : 0);                                     // spheres swept linearly
    info[6] = ds.n_fin - ds.n_arect - (bvh_f ? ds.n_fin_bvh : 0);                        // finite planes swept linearly
    info[7] = (int)((size_t)(ds.blob_f4 - ds.stage_off) * sizeof(float4));               // bytes staged per CTA
}

int tcrt_scene_structures(tcrt_ctx* ctx, int info[8]) {
    if (!ctx || !info) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    fill_structures(ctx->scene_ds, ctx->scene_grid, ctx->scene_bvh_s, ctx->scene_bvh_f, info);
    return TCRT_OK;
}

int tcrt_plan_grid_cells(const tcrt_scene* s, const float* points, int n_points, int* objects, int cap, int* counts,
                         float* grid_margin) {
    if (!s || !points || !counts || n_points < 0 || cap < 0 || (cap > 0 && !objects)) return fail(nullptr, TCRT_ERR_INVALID, "bad argument");
    if (int rc = validate_scene(nullptr, s)) return rc;
    SceneBlob b;
    const int rc = plan_scene_blob(s, b);
    if (rc) return fail(nullptr, rc, "%s", b.err.c_str());
    if (!b.grid) return fail(nullptr, TCRT_ERR_UNSUPPORTED, "the scene gets no sphere grid");
    const DeviceScene& ds = b.ds;
    if (grid_margin) *grid_margin = ds.grid_margin;
    const int* items = reinterpret_cast<const int*>(&b.host[b.off[8]]);
    const int* idx = reinterpret_cast<const int*>(&b.host[ds.idx_off]);
    for (int i = 0; i < n_points; i++) {
        const float* point = points + 3 * (size_t)i;
        int* out = objects + (size_t)i * cap;
        counts[i] = 0;
        int c[3];
        bool inside = true;
        for (int k = 0; k < 3; k++) {
            inside = inside && point[k] >= ds.grid_lo[k] && point[k] <= ds.grid_hi[k];
            // the kernel's own cell arithmetic (tcrt_render_grid.cu)
            c[k] = std::min(ds.grid_dims[k] - 1, std::max(0, (int)floorf((point[k] - ds.grid_lo[k]) * ds.grid_inv_cell[k])));
        }
        if (!inside) continue;                                                          // outside the grid's box
        const size_t cell = (size_t)c[0] + (size_t)ds.grid_dims[0] * ((size_t)c[1] + (size_t)ds.grid_dims[1] * c[2]);
        const float4 g = b.host[b.off[7] + 2 * cell];
        int meta[4];
        memcpy(meta, &b.host[b.off[7] + 2 * cell + 1], sizeof meta);
        int n = 0;
        if (g.w > 0.0f) {               // an empty cell carries the unhittable sphere (r^2 = -1e30)
            if (n < cap) out[n] = idx[meta[1]];
            n++;
            for (int j = 0; j < meta[0]; j++, n++)
                if (n < cap) out[n] = idx[items[meta[2] + j]];
        }
        counts[i] = n;
    }
    return TCRT_OK;
}

int tcrt_plan_scene(const tcrt_scene* s, int info[8], int grid_dims[3]) {
    if (!s || !info) return fail(nullptr, TCRT_ERR_INVALID, "null argument");
    if (int rc = validate_scene(nullptr, s)) return rc;
    SceneBlob b;
    const int rc = plan_scene_blob(s, b);
    if (rc) return fail(nullptr, rc, "%s", b.err.c_str());
    fill_structures(b.ds, b.grid, b.bvh_s, b.bvh_f, info);
    if (grid_dims)
        for (int k = 0; k < 3; k++) grid_dims[k] = b.grid ? b.ds.grid_dims[k] : 0;
    return TCRT_OK;
}

int tcrt_set_camera(tcrt_ctx* ctx, const tcrt_camera* cam) {
    if (!ctx || !cam) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    ctx->cam = *cam;
    ctx->cut_valid = false;
    ctx->costs_valid = false;
    return TCRT_OK;
}

static int check_full_frame(tcrt_ctx* ctx, const tcrt_params* p) {
    if (!ctx->has_frame) return fail(ctx, TCRT_ERR_NO_FRAME, "nothing rendered yet");
    if (ctx->frame_x0 != 0 || ctx->frame_x1 != p->width || ctx->frame_h != p->height)
        return fail(ctx, TCRT_ERR_INVALID, "last render covered columns [%d,%d) x %d, not the %dx%d image", ctx->frame_x0,
                    ctx->frame_x1, ctx->frame_h, p->width, p->height);
    return TCRT_OK;
}

static bool write_fully(int fd, const void* src, size_t n) {
    const char* s = static_cast<const char*>(src);
    while (n > 0) {
        ssize_t w = write(fd, s, n);
        if (w < 0 && errno == EINTR) continue;
        if (w <= 0) return false;
        s += w;
        n -= (size_t)w;
    }
    return true;
}

int tcrt_write_ppm(tcrt_ctx* ctx, const tcrt_params* p, const char* path) {
    if (!ctx || !p || !path) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    int rc = check_full_frame(ctx, p);
    if (rc) return rc;
    const size_t W = (size_t)p->width, H = (size_t)p->height;
    // every band is quantised AND turned into image rows on its device (the text scratch buffer doubles as the 8-bit
    // staging area); a strided copy drops it into its columns of the host image: no per-pixel work on the host
    std::vector<unsigned char> img(W * H * 3);
    for (auto& d : ctx->devs) {
        if (d.fr().x1 <= d.fr().x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        const size_t cols = (size_t)(d.fr().x1 - d.fr().x0);
        if (d.text_cap < cols * H * 3 + 16) {
            if (d.text) CK(ctx, cudaFree(d.text));
            d.text = nullptr;
            d.text_cap = 0;
            CK(ctx, cudaMalloc((void**)&d.text, cols * H * 3 + 16));
            d.text_cap = cols * H * 3 + 16;
        }
        ctx->txt_prepared = false;
        CK(ctx, tcrt_launch_quantize8_image(d.fr().frame, (int)cols, (int)H, reinterpret_cast<unsigned char*>(d.text), d.stream));
        CK(ctx, cudaMemcpy2DAsync(img.data() + (size_t)d.fr().x0 * 3, W * 3, d.text, cols * 3, cols * 3, H,
                                  cudaMemcpyDeviceToHost, d.stream));
    }
    for (auto& d : ctx->devs) {
        if (d.fr().x1 <= d.fr().x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));
    }
    char header[64];
    const int hn = snprintf(header, sizeof header, "P6\n%d %d\n255\n", p->width, p->height);
    int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0666);
    if (fd < 0) return fail(ctx, TCRT_ERR_IO, "Error Opening File %s", path);
    bool ok = write_fully(fd, header, (size_t)hn) && write_fully(fd, img.data(), img.size());
    ok = (close(fd) == 0) && ok;
    if (!ok) return fail(ctx, TCRT_ERR_IO, "short write to %s", path);
    return TCRT_OK;
}

int tcrt_write_bin(tcrt_ctx* ctx, const tcrt_params* p, const char* path) {
    if (!ctx || !p || !path) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    int rc = check_full_frame(ctx, p);
    if (rc) return rc;
    const size_t n = (size_t)p->width * p->height * 3;
    std::vector<float> host(n);
    rc = tcrt_download(ctx, host.data());
    if (rc) return rc;
    unsigned char header[32] = {'T', 'C', 'R', 'T', 'B', 'I', 'N', '1'};
    const int wh[2] = {p->width, p->height};
    memcpy(header + 8, wh, 8);
    int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0666);
    if (fd < 0) return fail(ctx, TCRT_ERR_IO, "Error Opening File %s", path);
    bool ok = write_fully(fd, header, sizeof header) && write_fully(fd, host.data(), n * sizeof(float));
    ok = (close(fd) == 0) && ok;
    if (!ok) return fail(ctx, TCRT_ERR_IO, "short write to %s", path);
    return TCRT_OK;
}

int tcrt_selftest_div3(tcrt_ctx* ctx, unsigned long long n_cases, unsigned int seed, unsigned long long* n_bad) {
    if (!ctx || !n_bad) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    DeviceState& d = ctx->devs[0];
    CK(ctx, cudaSetDevice(d.dev));
    CK(ctx, cudaMemsetAsync(d.fr().ctl, 0, 64, d.stream));
    CK(ctx, tcrt_launch_div3_check(n_cases, seed, reinterpret_cast<unsigned long long*>(d.fr().ctl), d.stream));
    CK(ctx, cudaMemcpyAsync(d.fr().h_counters, d.fr().ctl, 8, cudaMemcpyDeviceToHost, d.stream));
    CK(ctx, cudaStreamSynchronize(d.stream));
    *n_bad = d.fr().h_counters[0];
    return TCRT_OK;
}

// ---- .txt writer -----------------------------------------------------------------------------------
// Decide fixed/general per device and size the output.
static int prepare_txt(tcrt_ctx* ctx) {
    if (!ctx->has_frame) return fail(ctx, TCRT_ERR_NO_FRAME, "nothing rendered yet");
    if (ctx->txt_prepared) return TCRT_OK;
    for (auto& d : ctx->devs) {
        if (d.fr().x1 <= d.fr().x0) { d.txt_bytes = 0; continue; }
        CK(ctx, cudaSetDevice(d.dev));
        const size_t np = (size_t)(d.fr().x1 - d.fr().x0) * d.fr().height;
        CK(ctx, cudaMemsetAsync(d.flag, 0, 4, d.stream));
        CK(ctx, tcrt_launch_txt_fixed_check(d.fr().frame, np, d.flag, d.stream));
        CK(ctx, cudaMemcpyAsync(d.h_txt, d.flag, 4, cudaMemcpyDeviceToHost, d.stream));
    }
    for (auto& d : ctx->devs) {
        if (d.fr().x1 <= d.fr().x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));
        const size_t np = (size_t)(d.fr().x1 - d.fr().x0) * d.fr().height;
        d.txt_fixed = (*(volatile unsigned int*)d.h_txt) == 0u;
        if (d.txt_fixed) {
            d.txt_bytes = np * 31;
        } else {
            const size_t nb = (np + 255) / 256;
            int rc = ensure(ctx, d.offs, d.offs_cap, np);
            if (rc) return rc;
            rc = ensure(ctx, d.block_sums, d.bs_cap, nb + 1);
            if (rc) return rc;
            int launches = 0;
            CK(ctx, tcrt_launch_txt_lengths(d.fr().frame, np, d.offs, d.block_sums, d.stream, &launches));
            CK(ctx, cudaMemcpyAsync(d.h_txt + 1, d.block_sums + nb, 8, cudaMemcpyDeviceToHost, d.stream));
            CK(ctx, cudaStreamSynchronize(d.stream));
            d.txt_bytes = (size_t)d.h_txt[1];
        }
    }
    ctx->txt_prepared = true;
    return TCRT_OK;
}

int tcrt_txt_size(tcrt_ctx* ctx, size_t* n_bytes) {
    if (!ctx || !n_bytes) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    int rc = prepare_txt(ctx);
    if (rc) return rc;
    size_t t = 0;
    for (auto& d : ctx->devs) t += d.txt_bytes;
    *n_bytes = t;
    return TCRT_OK;
}

int tcrt_format_txt(tcrt_ctx* ctx, char* host_text, size_t cap, size_t* n_bytes) {
    if (!ctx || !host_text) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    size_t total = 0;
    int rc = tcrt_txt_size(ctx, &total);
    if (rc) return rc;
    if (total > cap) return fail(ctx, TCRT_ERR_INVALID, "text needs %zu bytes, buffer has %zu", total, cap);
    size_t off = 0;
    for (auto& d : ctx->devs) {
        if (d.fr().x1 <= d.fr().x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        const size_t np = (size_t)(d.fr().x1 - d.fr().x0) * d.fr().height;
        rc = ensure(ctx, d.text, d.text_cap, d.txt_bytes + 16);
        if (rc) return rc;
        if (d.txt_fixed) {
            CK(ctx, tcrt_launch_txt_fixed(d.fr().frame, np, d.text, d.stream));
        } else {
            CK(ctx, tcrt_launch_txt_general(d.fr().frame, np, d.offs, d.block_sums, d.text, d.stream));
        }
        CK(ctx, cudaMemcpyAsync(host_text + off, d.text, d.txt_bytes, cudaMemcpyDeviceToHost, d.stream));
        off += d.txt_bytes;
    }
    for (auto& d : ctx->devs) {
        if (d.fr().x1 <= d.fr().x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));
    }
    if (n_bytes) *n_bytes = total;
    return TCRT_OK;
}

int tcrt_format_pixels(tcrt_ctx* ctx, const float* host_rgb, size_t n_pixels, char* host_text, size_t cap,
                       size_t* n_bytes) {
    if (!ctx || (!host_rgb && n_pixels) || !host_text || !n_bytes) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    *n_bytes = 0;
    if (n_pixels == 0) return TCRT_OK;
    if (n_pixels > (size_t)0x7fffffff / 3) return fail(ctx, TCRT_ERR_INVALID, "too many pixels");
    DeviceState& d = ctx->devs[0];
    CK(ctx, cudaSetDevice(d.dev));
    // the frame buffer doubles as the staging area: the last render is gone afterwards
    ctx->has_frame = false;
    ctx->txt_prepared = false;
    int rc = ensure(ctx, d.fr().frame, d.fr().frame_cap, n_pixels * 3);
    if (rc) return rc;
    CK(ctx, cudaMemcpyAsync(d.fr().frame, host_rgb, n_pixels * 3 * sizeof(float), cudaMemcpyHostToDevice, d.stream));
    for (auto& o : ctx->devs) o.fr().x0 = o.fr().x1 = 0;
    d.fr().x0 = 0;
    d.fr().x1 = 1;                 // one "column" of n_pixels rows
    d.fr().height = (int)n_pixels;
    ctx->has_frame = true;
    ctx->frame_x0 = 0;
    ctx->frame_x1 = 1;
    ctx->frame_h = (int)n_pixels;
    rc = tcrt_format_txt(ctx, host_text, cap, n_bytes);
    ctx->has_frame = false;
    ctx->txt_prepared = false;
    return rc;
}

int tcrt_txt_header(const tcrt_params* p, double run_time_s, char* buf, size_t cap) {
    if (!p || !buf || cap == 0) return TCRT_ERR_INVALID;
    // init_log (RayTracer.cpp:2033-2058) then the three tags of printPixelsToLog (:1576-1578);
    // addToLogInt "%i", addToLogDouble "%f" (:2070-2096).  us/pixel = run_time_us / (W*H) with an
    // int product (:1577).
    const double us_per_pixel = (run_time_s * 1.0E6) / (p->width * p->height);
    int n = snprintf(buf, cap,
                     "OSX Awesome Picture\n"
                     "Horizontal_Resolution:%i.\n"
                     "Vertical_Resolution:%i.\n"
                     "Hardware_Target:OSX C++.\n"
                     "Number_of_Cores:%i.\n"
                     "IS_FOR_HARDWARE\n"
                     "NO_PARTIONING\n"
                     "Run_Time:%f.\n"
                     "us/pixel:%f.\n"
                     "filename:raytracer_screen.txt.\n",
                     p->width, p->height, 1, run_time_s, us_per_pixel);
    if (n < 0 || (size_t)n >= cap) return TCRT_ERR_INVALID;
    return n;
}

// ---- the file writer: format -> D2H -> page cache as a pipeline ----------------------------------------------
// Reference: printPixelsToLog (RayTracer.cpp:1574-1626) sprintf's and fputs's one pixel at a time after the
// render.  Here the pixel lines of a band are produced in chunks of 256 K pixels (7.9 MB of text): the GPU
// formats chunk k+1 while chunk k crosses the bus into pinned staging and worker threads copy finished chunks
// into the output file's mapping (mmap: page faults and copies of different chunks run on different cores; a
// write() per chunk would serialise on the inode lock).  Every pixel line whose channels are all in [0, 10) is
// exactly 31 bytes, so every chunk's place in the file is known beforehand; a frame with a longer line (rare:
// a channel >= 10, negative, inf/nan) is detected by the formatter's check kernel and takes the general path.
}  // extern "C"

namespace {

constexpr size_t kTxtLine = 31;
constexpr size_t kTxtChunkPx = 256 * 1024;
constexpr int kTxtSlots = 4;
constexpr int kTxtParts = 8;          // a chunk is copied into the file by up to this many workers at once

struct TxtSink {
    int fd = -1;
    char* map = nullptr;
    size_t size = 0;
    bool put(size_t off, const char* src, size_t n) const {
        if (map) {
            memcpy(map + off, src, n);
            return true;
        }
        while (n > 0) {
            ssize_t w = pwrite(fd, src, n, (off_t)off);
            if (w < 0 && errno == EINTR) continue;
            if (w <= 0) return false;
            src += w;
            off += (size_t)w;
            n -= (size_t)w;
        }
        return true;
    }
};

struct TxtPipe {
    struct Job {
        int dev;
        cudaEvent_t ev;
        const char* src;
        size_t off, n;
        std::atomic<int>* left;     // parts of this chunk still to copy; the slot is free at 0
        int* slot_busy;
    };
    std::mutex mu;
    std::condition_variable cv_job, cv_slot;
    std::deque<Job> jobs;
    bool closing = false;
    bool io_error = false;
    const TxtSink* sink = nullptr;
    std::vector<std::thread> workers;

    void start(const TxtSink* s, int n_workers) {
        sink = s;
        for (int i = 0; i < n_workers; i++) workers.emplace_back([this] { run(); });
    }
    void run() {
        int cur_dev = -1;
        for (;;) {
            Job j;
            {
                std::unique_lock<std::mutex> lk(mu);
                cv_job.wait(lk, [this] { return closing || !jobs.empty(); });
                if (jobs.empty()) return;
                j = jobs.front();
                jobs.pop_front();
            }
            if (cur_dev != j.dev) {
                cudaSetDevice(j.dev);
                cur_dev = j.dev;
            }
            const bool ok = cudaEventSynchronize(j.ev) == cudaSuccess && sink->put(j.off, j.src, j.n);
            std::lock_guard<std::mutex> lk(mu);
            if (!ok) io_error = true;
            if (j.left->fetch_sub(1) == 1) {
                *j.slot_busy = 0;
                cv_slot.notify_all();
            }
        }
    }
    void push(const Job& j) {
        {
            std::lock_guard<std::mutex> lk(mu);
            jobs.push_back(j);
        }
        cv_job.notify_one();
    }
    void wait_slot(int* slot_busy) {
        std::unique_lock<std::mutex> lk(mu);
        cv_slot.wait(lk, [slot_busy] { return *slot_busy == 0; });
    }
    void finish() {
        {
            std::lock_guard<std::mutex> lk(mu);
            closing = true;
        }
        cv_job.notify_all();
        for (auto& t : workers) t.join();
        workers.clear();
    }
};

// Pixel lines of device d's band of the last render, fixed-width layout, into `sink` at byte `base` + (pixel
// index within the whole image) * 31.  *not_fixed != 0 afterwards: some line is longer, the bytes are void.
int stream_band_fixed(tcrt_ctx* ctx, DeviceState& d, TxtPipe& pipe, size_t base, unsigned int* not_fixed, std::string* err) {
    auto cuda_fail = [&](const char* what, cudaError_t e) {
        *err = std::string(what) + ": " + cudaGetErrorString(e);
        return TCRT_ERR_CUDA;
    };
    FrameRes& f = d.fr();
    *not_fixed = 0;
    if (f.x1 <= f.x0) return TCRT_OK;
    cudaError_t e = cudaSetDevice(d.dev);
    if (e != cudaSuccess) return cuda_fail("cudaSetDevice", e);
    const size_t np = (size_t)(f.x1 - f.x0) * f.height;
    const size_t chunk_bytes = kTxtChunkPx * kTxtLine;
    if (d.text_cap < kTxtSlots * chunk_bytes) {
        if (d.text) cudaFree(d.text);
        d.text = nullptr;
        d.text_cap = 0;
        if ((e = cudaMalloc((void**)&d.text, kTxtSlots * chunk_bytes)) != cudaSuccess) return cuda_fail("cudaMalloc(text)", e);
        d.text_cap = kTxtSlots * chunk_bytes;
    }
    if (!d.txt_stage) {
        if ((e = cudaHostAlloc((void**)&d.txt_stage, kTxtSlots * chunk_bytes, cudaHostAllocPortable)) != cudaSuccess)
            return cuda_fail("cudaHostAlloc(txt staging)", e);
        for (auto& ev : d.ev_txt)
            if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return cuda_fail("cudaEventCreate", e);
    }
    if ((e = cudaMemsetAsync(d.flag, 0, 4, d.stream)) != cudaSuccess) return cuda_fail("cudaMemsetAsync", e);
    int slot_busy[kTxtSlots] = {};
    std::atomic<int> left[kTxtSlots];
    for (auto& l : left) l.store(0);
    const size_t first_px = (size_t)f.x0 * f.height;     // x-major: the band is one run of pixel lines
    int rc = TCRT_OK;
    size_t c = 0;
    for (size_t p0 = 0; p0 < np && rc == TCRT_OK; p0 += kTxtChunkPx, c++) {
        const int slot = (int)(c % kTxtSlots);
        const size_t n = std::min(kTxtChunkPx, np - p0);
        pipe.wait_slot(&slot_busy[slot]);
        char* dtext = d.text + slot * chunk_bytes;
        char* stage = d.txt_stage + slot * chunk_bytes;
        if ((e = tcrt_launch_txt_fixed_check(f.frame + 3 * p0, n, d.flag, d.stream)) != cudaSuccess ||
            (e = tcrt_launch_txt_fixed(f.frame + 3 * p0, n, dtext, d.stream)) != cudaSuccess ||
            (e = cudaMemcpyAsync(stage, dtext, n * kTxtLine, cudaMemcpyDeviceToHost, d.stream)) != cudaSuccess ||
            (e = cudaEventRecord(d.ev_txt[slot], d.stream)) != cudaSuccess) {
            rc = cuda_fail("txt chunk", e);
            break;
        }
        const size_t bytes = n * kTxtLine;
        const int parts = bytes >= (size_t)kTxtParts * 65536 ? kTxtParts : 1;
        slot_busy[slot] = 1;
        left[slot].store(parts);
        for (int k = 0; k < parts; k++) {
            const size_t b0 = bytes * k / parts, b1 = bytes * (k + 1) / parts;
            pipe.push({d.dev, d.ev_txt[slot], stage + b0, base + (first_px + p0) * kTxtLine + b0, b1 - b0, &left[slot], &slot_busy[slot]});
        }
    }
    for (int sl = 0; sl < kTxtSlots; sl++) pipe.wait_slot(&slot_busy[sl]);
    if (rc) return rc;
    if ((e = cudaMemcpyAsync(d.h_txt, d.flag, 4, cudaMemcpyDeviceToHost, d.stream)) != cudaSuccess ||
        (e = cudaStreamSynchronize(d.stream)) != cudaSuccess)
        return cuda_fail("txt flag", e);
    *not_fixed = *(volatile unsigned int*)d.h_txt;
    return TCRT_OK;
}

int n_txt_workers() {
    const unsigned hc = std::thread::hardware_concurrency();
    return (int)std::max(2u, std::min(16u, hc ? hc : 4u));
}

// The pinned staging slots of one device that a staged copy cycles through, and which of them still hold bytes on their way
// to the destination.
struct StageSlots {
    int busy[kTxtSlots] = {};
    std::atomic<int> left[kTxtSlots];
    size_t piece = 0;
    StageSlots() {
        for (auto& l : left) l.store(0);
    }
    void drain(TxtPipe& pipe) {
        for (int sl = 0; sl < kTxtSlots; sl++) pipe.wait_slot(&busy[sl]);
    }
};

// Device d's pinned staging slots (shared with the .txt writer), allocated at first use.
cudaError_t ensure_stage(DeviceState& d) {
    cudaError_t e = cudaSuccess;
    if (!d.txt_stage) {
        e = cudaHostAlloc((void**)&d.txt_stage, kTxtSlots * kTxtChunkPx * kTxtLine, cudaHostAllocPortable);
        for (auto& ev : d.ev_txt)
            if (e == cudaSuccess) e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    }
    return e;
}

// n bytes of device memory at src -> byte dst of the copy sink: on d's copy stream once `ready` has completed (nullptr: the
// bytes are complete already), slot by slot into d's pinned staging at bus speed, from there by the pipe's worker threads.
// The caller has called cudaSetDevice(d.dev) and ensure_stage(d), and drains `slots` before the destination may be read.
cudaError_t stage_out(TxtPipe& pipe, DeviceState& d, StageSlots& slots, const char* src, size_t n, size_t dst, cudaEvent_t ready) {
    const size_t slot_bytes = kTxtChunkPx * kTxtLine;
    cudaError_t e = ready ? cudaStreamWaitEvent(d.copy_stream, ready, 0) : cudaSuccess;
    for (size_t b = 0; b < n && e == cudaSuccess; b += slot_bytes, slots.piece++) {
        const int slot = (int)(slots.piece % kTxtSlots);
        const size_t m = std::min(slot_bytes, n - b);
        pipe.wait_slot(&slots.busy[slot]);
        char* stage = d.txt_stage + slot * slot_bytes;
        e = cudaMemcpyAsync(stage, src + b, m, cudaMemcpyDeviceToHost, d.copy_stream);
        if (e == cudaSuccess) e = cudaEventRecord(d.ev_txt[slot], d.copy_stream);
        if (e != cudaSuccess) break;
        const int parts = m >= (size_t)kTxtParts * 65536 ? kTxtParts : 1;
        slots.busy[slot] = 1;
        slots.left[slot].store(parts);
        for (int q = 0; q < parts; q++) {
            const size_t b0 = m * q / parts, b1 = m * (q + 1) / parts;
            pipe.push({d.dev, d.ev_txt[slot], stage + b0, dst + b + b0, b1 - b0, &slots.left[slot], &slots.busy[slot]});
        }
    }
    return e;
}

}  // namespace

// The staged copy's worker threads, now writing into host (their sink).
static TxtPipe& copy_pipe_to(tcrt_ctx* ctx, void* host) {
    if (!ctx->copy_pipe) {      // the workers live as long as the ctx: starting eight threads costs as much as a 1080p frame
        ctx->copy_sink = new TxtSink();
        ctx->copy_pipe = new TxtPipe();
        ctx->copy_pipe->start(ctx->copy_sink, std::min(8, n_txt_workers()));
    }
    ctx->copy_sink->map = reinterpret_cast<char*>(host);     // the workers are idle between calls
    ctx->copy_pipe->io_error = false;
    return *ctx->copy_pipe;
}

// The band of the frame just submitted with kCopyStaged -> pageable host memory: chunk after chunk (as their kernels
// finish) into the pinned staging slots of the .txt writer at bus speed, from there by worker threads into host_band.
// fmt picks the device buffer (float frame or its 8-bit copy) and the bytes per pixel.
static int copy_out_staged(tcrt_ctx* ctx, const tcrt_params* p, int x0, void* host_band, FrameFormat fmt) {
    const size_t bpp = bytes_per_px(fmt);
    TxtPipe& pipe = copy_pipe_to(ctx, host_band);
    int rc = TCRT_OK;
    std::string err;
    for (auto& d : ctx->devs) {
        FrameRes& f = d.fr();
        if (f.x1 <= f.x0 || rc) continue;
        cudaError_t e = cudaSetDevice(d.dev);
        if (e == cudaSuccess) e = ensure_stage(d);
        StageSlots slots;
        // chunk k may leave once its kernel has finished (a frame that is already complete — tcrt_download — has no chunk
        // events of its own: older ones have long completed, and the render call has waited for the frame)
        const int n_chunks = std::max(1, f.n_chunks);
        for (int k = 0; k < n_chunks && e == cudaSuccess; k++) {
            const int cx0 = f.n_chunks ? f.chunk_x[k] : f.x0, cx1 = f.n_chunks ? f.chunk_x[k + 1] : f.x1;
            const size_t c0 = (size_t)(cx0 - f.x0) * p->height * bpp, c1 = (size_t)(cx1 - f.x0) * p->height * bpp;
            if (c1 <= c0) continue;
            // every chunk, the only one of a band too (a device band of a multi-device frame can be a single chunk although
            // the frame is large enough to be staged): the copy stream is not ordered behind the render streams otherwise
            e = stage_out(pipe, d, slots, frame_src(f, fmt) + c0, c1 - c0, (size_t)(f.x0 - x0) * p->height * bpp + c0,
                          f.n_chunks ? f.ev_chunk[k] : nullptr);
        }
        slots.drain(pipe);
        if (e != cudaSuccess) {
            err = cudaGetErrorString(e);
            rc = TCRT_ERR_CUDA;
        }
    }
    if (rc == TCRT_OK && pipe.io_error) {
        err = "a chunk did not arrive";
        rc = TCRT_ERR_CUDA;
    }
    return rc ? fail(ctx, rc, "staged copy-out: %s", err.c_str()) : TCRT_OK;
}

static void destroy_copy_pipe(tcrt_ctx* ctx) {
    if (ctx->copy_pipe) {
        ctx->copy_pipe->finish();
        delete ctx->copy_pipe;
        delete ctx->copy_sink;
        ctx->copy_pipe = nullptr;
        ctx->copy_sink = nullptr;
    }
}

// ---- primary-hit buffers and picking (tcrt_hits.cu) -------------------------------------------------------------------
// What the hit kernel needs of the frame p over columns [cx0, cx1) of device d: its rays are the render's primary rays.
static HitLaunch hit_launch(tcrt_ctx* ctx, DeviceState& d, const tcrt_params* p, int cx0, int cx1, unsigned int* queue) {
    HitLaunch hl{};
    RenderLaunch& rl = hl.rl;
    rl.scene = d.ds;
    rl.cam = ctx->cam;
    rl.width = p->width;
    rl.height = p->height;
    rl.x0 = cx0;
    rl.x1 = cx1;
    rl.far_dist = p->far_dist;
    rl.n_objects = ctx->n_objects;
    rl.queue = queue;
    return hl;
}

// A plain malloc'd / numpy destination, which cudaMemcpyAsync copies into at the driver's staging rate (render_impl).
static bool host_pageable(const void* p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return at.type == cudaMemoryTypeUnregistered;
}

extern "C" {

int tcrt_hit_buffers(tcrt_ctx* ctx, const tcrt_params* p, int x0, int x1, int* host_object, float* host_distance,
                     float* host_normal, tcrt_stats* stats) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null ctx");
    if (!valid_params(p)) return fail(ctx, TCRT_ERR_INVALID, "bad params");
    if (x0 < 0 || x1 > p->width || x0 >= x1) return fail(ctx, TCRT_ERR_INVALID, "bad column range [%d,%d)", x0, x1);
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    const int nd = (int)ctx->devs.size();
    const int h = p->height;
    // one band of equal width per device: every pixel costs one sweep, so there is nothing to balance
    std::vector<int> cut(nd + 1);
    for (int i = 0; i <= nd; i++) cut[i] = x0 + (int)((long long)(x1 - x0) * i / nd);
    // the three buffers: destination, bytes per pixel, word offset per pixel of the band in hit_mem
    char* host[3] = {reinterpret_cast<char*>(host_object), reinterpret_cast<char*>(host_distance),
                     reinterpret_cast<char*>(host_normal)};
    const size_t bpp[3] = {4, 4, 12}, word_off[3] = {0, 1, 2};
    // pageable destinations of at least 512 K pixels go through the pinned staging, as frames do (render_impl)
    const bool big = (long long)(x1 - x0) * h >= 512 * 1024;
    bool staged[3], any_direct = false;
    for (int k = 0; k < 3; k++) {
        staged[k] = host[k] && big && host_pageable(host[k]);
        any_direct = any_direct || (host[k] && !staged[k]);
    }
    ctx->has_hits = false;
    int launches = 0;
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        d.hit_x0 = cut[i];
        d.hit_x1 = cut[i + 1];
        d.hit_h = h;
        if (d.hit_x1 <= d.hit_x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        const size_t n = (size_t)(d.hit_x1 - d.hit_x0) * h;
        const int rc = ensure(ctx, d.hit_mem, d.hit_mem_cap, 5 * n);
        if (rc) return rc;
        HitLaunch hl = hit_launch(ctx, d, p, d.hit_x0, d.hit_x1, d.hit_queue);
        hl.object = reinterpret_cast<int*>(d.hit_mem);
        hl.distance = d.hit_mem + n;
        hl.normal = d.hit_mem + 2 * n;
        // on the render stream, behind whatever is queued there (a scene upload, frames in flight)
        CK(ctx, cudaMemsetAsync(d.hit_queue, 0, 4, d.stream));
        CK(ctx, cudaEventRecord(d.ev_h0, d.stream));
        CK(ctx, tcrt_launch_hits(hl, d.sm_count, d.stream));
        launches++;
        CK(ctx, cudaEventRecord(d.ev_h1, d.stream));
        if (any_direct) {
            CK(ctx, cudaStreamWaitEvent(d.copy_stream, d.ev_h1, 0));
            for (int k = 0; k < 3; k++)
                if (host[k] && !staged[k])
                    CK(ctx, cudaMemcpyAsync(host[k] + (size_t)(d.hit_x0 - x0) * h * bpp[k], d.hit_mem + word_off[k] * n,
                                            n * bpp[k], cudaMemcpyDeviceToHost, d.copy_stream));
            CK(ctx, cudaEventRecord(d.ev_hc, d.copy_stream));
        }
    }
    for (int k = 0; k < 3; k++) {
        if (!staged[k]) continue;
        TxtPipe& pipe = copy_pipe_to(ctx, host[k]);
        cudaError_t e = cudaSuccess;
        for (auto& d : ctx->devs) {
            if (d.hit_x1 <= d.hit_x0) continue;
            const size_t n = (size_t)(d.hit_x1 - d.hit_x0) * h;
            e = cudaSetDevice(d.dev);
            if (e == cudaSuccess) e = ensure_stage(d);
            StageSlots slots;
            if (e == cudaSuccess)
                e = stage_out(pipe, d, slots, reinterpret_cast<const char*>(d.hit_mem + word_off[k] * n), n * bpp[k],
                              (size_t)(d.hit_x0 - x0) * h * bpp[k], d.ev_h1);
            slots.drain(pipe);
            if (e != cudaSuccess) break;
        }
        if (e != cudaSuccess || pipe.io_error)
            return fail(ctx, TCRT_ERR_CUDA, "staged copy-out of a hit buffer: %s",
                        e != cudaSuccess ? cudaGetErrorString(e) : "a chunk did not arrive");
    }
    if (stats) memset(stats, 0, sizeof(*stats));
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        if (stats) {
            stats->col_begin[i] = d.hit_x0;
            stats->col_end[i] = d.hit_x1;
        }
        if (d.hit_x1 <= d.hit_x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaEventSynchronize(d.ev_h1));
        if (any_direct) CK(ctx, cudaEventSynchronize(d.ev_hc));
        if (stats) {
            float ms = 0.f;
            CK(ctx, cudaEventElapsedTime(&ms, d.ev_h0, d.ev_h1));
            stats->render_ms[i] = ms;
            if (any_direct) CK(ctx, cudaEventElapsedTime(&ms, d.ev_h1, d.ev_hc));
            stats->d2h_ms[i] = any_direct ? std::max(ms, 0.f) : 0.0;   // copy time not hidden behind the kernel
            stats->rays_primary[i] = (unsigned long long)(d.hit_x1 - d.hit_x0) * h;
        }
    }
    if (stats) {
        stats->n_devices = nd;
        stats->gpu_launches = (unsigned long long)launches;
    }
    ctx->has_hits = true;
    return TCRT_OK;
}

int tcrt_device_hit_buffers(tcrt_ctx* ctx, int slot, int** object, float** distance, float** normal, size_t* n_pixels) {
    if (!ctx || slot < 0 || slot >= (int)ctx->devs.size() || !object || !distance || !normal || !n_pixels)
        return fail(ctx, TCRT_ERR_INVALID, "bad argument");
    if (!ctx->has_hits) return fail(ctx, TCRT_ERR_NO_FRAME, "no hit buffers computed yet");
    DeviceState& d = ctx->devs[slot];
    const size_t n = d.hit_x1 > d.hit_x0 ? (size_t)(d.hit_x1 - d.hit_x0) * d.hit_h : 0;
    *object = n ? reinterpret_cast<int*>(d.hit_mem) : nullptr;
    *distance = n ? d.hit_mem + n : nullptr;
    *normal = n ? d.hit_mem + 2 * n : nullptr;
    *n_pixels = n;
    return TCRT_OK;
}

int tcrt_pick(tcrt_ctx* ctx, const tcrt_params* p, int n, const int* xz, int* object, float* distance, float* normal) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null ctx");
    if (!valid_params(p)) return fail(ctx, TCRT_ERR_INVALID, "bad params");
    if (n < 0 || (n > 0 && !xz)) return fail(ctx, TCRT_ERR_INVALID, "bad pixel list");
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    for (int i = 0; i < n; i++)
        if (xz[2 * i] < 0 || xz[2 * i] >= p->width || xz[2 * i + 1] < 0 || xz[2 * i + 1] >= p->height)
            return fail(ctx, TCRT_ERR_INVALID, "pick %d: pixel (%d, %d) outside the %dx%d frame", i, xz[2 * i], xz[2 * i + 1],
                        p->width, p->height);
    if (n == 0) return TCRT_OK;
    DeviceState& d = ctx->devs[0];
    CK(ctx, cudaSetDevice(d.dev));
    const size_t m = (size_t)n;
    const int rc = ensure(ctx, d.pick_mem, d.pick_mem_cap, 7 * m);
    if (rc) return rc;
    HitLaunch hl = hit_launch(ctx, d, p, 0, p->width, d.hit_queue + 1);
    hl.xz = d.pick_mem;
    hl.n_list = n;
    hl.object = d.pick_mem + 2 * m;
    hl.distance = reinterpret_cast<float*>(d.pick_mem + 3 * m);
    hl.normal = reinterpret_cast<float*>(d.pick_mem + 4 * m);
    CK(ctx, cudaMemcpyAsync(d.pick_mem, xz, 2 * m * sizeof(int), cudaMemcpyHostToDevice, d.stream));
    CK(ctx, cudaMemsetAsync(d.hit_queue + 1, 0, 4, d.stream));
    CK(ctx, tcrt_launch_hits(hl, d.sm_count, d.stream));
    if (object) CK(ctx, cudaMemcpyAsync(object, hl.object, m * sizeof(int), cudaMemcpyDeviceToHost, d.stream));
    if (distance) CK(ctx, cudaMemcpyAsync(distance, hl.distance, m * sizeof(float), cudaMemcpyDeviceToHost, d.stream));
    if (normal) CK(ctx, cudaMemcpyAsync(normal, hl.normal, 3 * m * sizeof(float), cudaMemcpyDeviceToHost, d.stream));
    CK(ctx, cudaEventRecord(d.ev_h1, d.stream));
    CK(ctx, cudaEventSynchronize(d.ev_h1));
    return TCRT_OK;
}

}  // extern "C"

// ---- ray batches (tcrt_trace_rays, tcrt_intersect_rays): the render and hit kernels' ray mode ---------------------------
// Rays per piece: 4 Mi keeps every kernel index far inside int; a piece's scratch is 4 Mi * 11 words = 176 MB at most.
constexpr size_t kRayPiece = (size_t)1 << 22;

// The ray-batch events and control block of device d, created at first use.
static int ensure_ray_state(tcrt_ctx* ctx, DeviceState& d) {
    if (d.ray_ctl) return TCRT_OK;
    for (int si = 0; si < kChunkStreams; si++) {
        CK(ctx, cudaEventCreateWithFlags(&d.ev_rk[si], cudaEventDisableTiming));
        CK(ctx, cudaEventCreateWithFlags(&d.ev_rin[si], cudaEventDisableTiming));
        CK(ctx, cudaEventCreateWithFlags(&d.ev_rout[si], cudaEventDisableTiming));
    }
    CK(ctx, cudaEventCreate(&d.ev_r0));
    CK(ctx, cudaEventCreate(&d.ev_r1));
    CK(ctx, cudaEventCreate(&d.ev_rc));
    CK(ctx, cudaHostAlloc((void**)&d.h_ray, 64 * kChunkStreams, cudaHostAllocPortable));
    CK(ctx, cudaMalloc((void**)&d.ray_ctl, 64 * kChunkStreams));
    return TCRT_OK;
}

// Pinned host memory of at least `need` floats in p (its contents are not kept).
static int ensure_pinned(tcrt_ctx* ctx, float*& p, size_t& cap, size_t need) {
    if (need <= cap && p) return TCRT_OK;
    if (p) CK(ctx, cudaFreeHost(p));
    p = nullptr;
    cap = 0;
    CK(ctx, cudaHostAlloc((void**)&p, need * sizeof(float), cudaHostAllocPortable));
    cap = need;
    return TCRT_OK;
}

// Is p device memory of device dev?
static bool on_device(const void* p, int dev) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice && at.device == dev;
}

// What a batch computes: the colour of each ray (render kernels' ray mode), its nearest hit (hit kernel's ray mode),
// whether it is occluded before its limit, whether each point is occluded from each light (occlusion kernel), or the
// columns of a stack of views (render kernels' views mode; an item is one global column of height pixels).
enum BatchKind { kBatchColour, kBatchHits, kBatchOccRays, kBatchOccPoints, kBatchViews };

// One batch: [0, n) split into equal contiguous ranges, one per device (device forms: slot only), each run in pieces round
// robin over the render streams: at most kRayPiece rays, or (points) kRayPiece (point, light) pairs and at least one point.
// A piece of a host form is: its inputs to the stream's scratch (pinned ones straight, pageable ones through the stream's
// pinned staging), one launch, its outputs to the host on the copy stream (pinned ones straight, pageable ones through
// stage_out).  A piece's outputs are sent once the next piece has been queued, so a piece's copies overlap other pieces'
// launches; a stream's next piece waits for them before it reuses the scratch.  Device forms launch on the caller's buffers
// directly.  Inputs: directions (rays) or points, origins (rays), tmax (occluded rays).  out[0] rgb (colour), object (hits)
// or the occlusion bytes, out[1] distance, out[2] normal (hits).  p: params of the colour and hit kinds, nullptr otherwise.
// Views: n = n_views * width global columns; the only input is the camera table `cams` (n / width cameras, copied once per
// device to its view_cams before the first piece); out[0] rgb, out[1] rgb8, either may be nullptr.  Pieces are at most
// kRayPiece pixels, whole columns, multiples of 4 columns when width % 4 == 0 (and the pieces hold at least 4), and so is
// the cut between devices.  A piece is one views launch into the float scratch (device form: into rgb in place, or the
// scratch when only rgb8 is requested), then for rgb8 one quantisation launch on the same stream.
static int rays_impl(tcrt_ctx* ctx, int slot, BatchKind kind, const tcrt_params* p, size_t n, const float* origins,
                     int shared_origin, const float* dirs, const float* tmax, void* const out_in[3],
                     unsigned long long* n_invalid, tcrt_stats* stats, const tcrt_camera* cams = nullptr) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null ctx");
    const bool hits = kind == kBatchHits, occ = kind == kBatchOccRays || kind == kBatchOccPoints;
    const bool points = kind == kBatchOccPoints, views = kind == kBatchViews;
    if (!occ && !p) return fail(ctx, TCRT_ERR_INVALID, "null params");
    const bool device_form = slot >= 0;
    if (device_form && slot >= (int)ctx->devs.size()) return fail(ctx, TCRT_ERR_INVALID, "device slot %d out of range", slot);
    if (kind == kBatchColour && p->max_depth < 0) return fail(ctx, TCRT_ERR_INVALID, "max_depth %d < 0", p->max_depth);
    char* out[3] = {static_cast<char*>(out_in[0]), static_cast<char*>(out_in[1]), static_cast<char*>(out_in[2])};
    if (hits ? (!out[0] && !out[1] && !out[2]) : views ? (!out[0] && !out[1]) : !out[0])
        return fail(ctx, TCRT_ERR_INVALID, "no output");
    if (n > 0 && (views ? !cams : points ? !dirs : (!origins || !dirs || (kind == kBatchOccRays && !tmax))))
        return fail(ctx, TCRT_ERR_INVALID, views ? "null cameras" : "null ray input");
    if (views && !valid_params(p)) return fail(ctx, TCRT_ERR_INVALID, "bad params");
    if (n > SIZE_MAX / (6 * sizeof(float))) return fail(ctx, TCRT_ERR_INVALID, "%zu rays: byte count overflows", n);
    if ((kind == kBatchColour || views) && p->max_depth > TCRT_MAX_DEPTH)
        return fail(ctx, TCRT_ERR_UNSUPPORTED, "max_depth %d > TCRT_MAX_DEPTH %d", p->max_depth, TCRT_MAX_DEPTH);
    if (device_form && n > 0) {
        const int dev = ctx->devs[slot].dev;
        const void* ptrs[6] = {origins, dirs, tmax, out[0], out[1], out[2]};
        for (const void* q : ptrs)
            if (q && !on_device(q, dev))
                return fail(ctx, TCRT_ERR_INVALID, "pointer %p is not device memory of device %d (slot %d)", q, dev, slot);
    }
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    // output bytes per point (a scene without lights: nothing to answer, nothing launched)
    const size_t n_lights = points ? (size_t)ctx->devs[0].ds.n_lights : 1;
    if (n_lights > 0 && n > SIZE_MAX / n_lights)
        return fail(ctx, TCRT_ERR_INVALID, "%zu points x %zu lights: byte count overflows", n, n_lights);
    tcrt_params occ_params;   // read by band_launch only; the occlusion kernel reads none of it
    if (occ) {
        tcrt_default_params(&occ_params);
        p = &occ_params;
    }
    const int nd = (int)ctx->devs.size();
    const int d_begin = device_form ? slot : 0, d_end = device_form ? slot + 1 : nd;
    // views: devices and pieces are cut on multiples of 4 columns when the views' width is (whole 4x8 tiles)
    const size_t unit = views && p->width % TCRT_TILE_W == 0 ? TCRT_TILE_W : 1;
    std::vector<size_t> cut(nd + 1, 0);
    for (int i = 0; i <= nd; i++)
        cut[i] = device_form ? (i <= slot ? 0 : n) : (n / unit / nd * i + n / unit % nd * i / nd) * unit;
    // inputs, in the order of the scratch: directions or points (3 floats per item), origins (3 per item, or 3 in all when
    // shared), tmax (1 per item); views have none (their camera table is copied once, not per piece)
    const int n_in = views ? 0 : kind == kBatchOccRays ? 3 : points ? 1 : 2;
    const float* in_src[3] = {dirs, origins, tmax};
    auto in_words = [&](int k, size_t cnt) -> size_t { return k == 1 ? (shared_origin ? 3 : 3 * cnt) : (k == 0 ? 3 : 1) * cnt; };
    // bytes per item of each output
    const int n_out = hits ? 3 : views ? 2 : 1;
    const size_t col_px = views ? (size_t)p->height : 1;   // pixels per item
    const size_t out_bytes[3] = {hits ? (size_t)4 : occ ? n_lights : 12 * col_px, views ? 3 * col_px : 4, 12};
    const size_t item_out = out_bytes[0] + (hits ? out_bytes[1] + out_bytes[2] : views ? out_bytes[1] : 0);
    bool staged[3] = {false, false, false}, any_direct = false;
    bool in_pageable[3] = {false, false, false}, any_pageable = false;
    if (!device_form && n > 0) {
        for (int k = 0; k < n_out; k++) {
            staged[k] = out[k] && host_pageable(out[k]);
            any_direct = any_direct || (out[k] && !staged[k]);
        }
        for (int k = 0; k < n_in; k++) any_pageable = any_pageable || (in_pageable[k] = host_pageable(in_src[k]));
    }
    if (stats) memset(stats, 0, sizeof(*stats));
    if (n_invalid) *n_invalid = 0;
    auto stream_of = [](DeviceState& d, int si) { return si == 0 ? d.stream : d.chunk_stream[si - 1]; };
    std::vector<int> used_streams(nd, 0), launches(nd, 0);
    size_t piece_items = std::max<size_t>(1, kRayPiece / std::max<size_t>(1, n_lights) / col_px);
    if (piece_items >= unit) piece_items -= piece_items % unit;
    for (int i = d_begin; i < d_end; i++) {
        DeviceState& d = ctx->devs[i];
        const size_t r0 = cut[i], r1 = cut[i + 1];
        if (r1 <= r0 || n_lights == 0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        int rc = ensure_ray_state(ctx, d);
        if (rc) return rc;
        const size_t n_pieces = (r1 - r0 + piece_items - 1) / piece_items;
        const int ns = ctx->one_stream ? 1 : (int)std::min<size_t>(kChunkStreams, n_pieces);
        used_streams[i] = ns;
        const size_t per = std::min(piece_items, r1 - r0);
        // scratch: the inputs, then the outputs (hits: object, distance, normal)
        auto all_in = [&](size_t cnt) {
            size_t w = 0;
            for (int k = 0; k < n_in; k++) w += in_words(k, cnt);
            return w;
        };
        if (!device_form) {
            for (int si = 0; si < ns; si++)
                if ((rc = ensure(ctx, d.ray_mem[si], d.ray_mem_cap[si], all_in(per) + (per * item_out + 3) / 4))) return rc;
            if (any_pageable)
                for (int si = 0; si < ns; si++)
                    if ((rc = ensure_pinned(ctx, d.ray_stage[si], d.ray_stage_cap[si], all_in(per)))) return rc;
        } else if (views && !out[0]) {   // rgb8 only: the floats go to the scratch
            for (int si = 0; si < ns; si++)
                if ((rc = ensure(ctx, d.ray_mem[si], d.ray_mem_cap[si], per * col_px * 3))) return rc;
        }
        // on the render stream, behind whatever is queued there (a scene upload, frames in flight); the other render
        // streams start behind it
        if (views) {
            const size_t n_cams = n / (size_t)p->width;
            if ((rc = ensure(ctx, d.view_cams, d.view_cams_cap, n_cams))) return rc;
            CK(ctx, cudaMemcpyAsync(d.view_cams, cams, n_cams * sizeof(tcrt_camera), cudaMemcpyHostToDevice, d.stream));
        }
        CK(ctx, cudaMemsetAsync(d.ray_ctl, 0, 64 * ns, d.stream));
        CK(ctx, cudaEventRecord(d.ev_r0, d.stream));
        for (int si = 1; si < ns; si++) CK(ctx, cudaStreamWaitEvent(stream_of(d, si), d.ev_r0, 0));
        // piece k: items [r0 + k*per, ...) on stream k % ns
        auto piece = [&](size_t k, size_t& a, size_t& cnt, int& si) {
            a = r0 + k * per;
            cnt = std::min(per, r1 - a);
            si = (int)(k % (size_t)ns);
        };
        auto out_dev = [&](int si, size_t cnt, int k) -> char* {   // output k of a piece in the stream's scratch
            char* base = reinterpret_cast<char*>(d.ray_mem[si] + all_in(cnt));
            return base + (k == 0 ? 0 : k == 1 ? cnt * out_bytes[0] : cnt * (out_bytes[0] + out_bytes[1]));
        };
        auto send_out = [&](size_t k) -> int {
            size_t a, cnt;
            int si;
            piece(k, a, cnt, si);
            if (any_direct) {
                CK(ctx, cudaStreamWaitEvent(d.copy_stream, d.ev_rk[si], 0));
                for (int b = 0; b < n_out; b++)
                    if (out[b] && !staged[b])
                        CK(ctx, cudaMemcpyAsync(out[b] + a * out_bytes[b], out_dev(si, cnt, b), cnt * out_bytes[b],
                                                cudaMemcpyDeviceToHost, d.copy_stream));
            }
            for (int b = 0; b < n_out; b++) {
                if (!staged[b]) continue;
                CK(ctx, ensure_stage(d));
                TxtPipe& pipe = copy_pipe_to(ctx, out[b]);
                StageSlots slots;
                const cudaError_t e = stage_out(pipe, d, slots, out_dev(si, cnt, b), cnt * out_bytes[b], a * out_bytes[b],
                                                d.ev_rk[si]);
                slots.drain(pipe);
                if (e != cudaSuccess || pipe.io_error)
                    return fail(ctx, TCRT_ERR_CUDA, "staged copy-out of a ray batch: %s",
                                e != cudaSuccess ? cudaGetErrorString(e) : "a chunk did not arrive");
            }
            CK(ctx, cudaEventRecord(d.ev_rout[si], d.copy_stream));
            return TCRT_OK;
        };
        const size_t lag = (!device_form && ns > 1) ? 1 : 0;
        for (size_t k = 0; k < n_pieces + lag; k++) {
            if (k < n_pieces) {
                size_t a, cnt;
                int si;
                piece(k, a, cnt, si);
                const cudaStream_t ks = stream_of(d, si);
                const float* src[3];
                for (int b = 0; b < n_in; b++)
                    src[b] = in_src[b] + (b == 1 && shared_origin ? 0 : in_words(b, a));
                void* dst[3] = {out[0], out[1], out[2]};
                if (!device_form) {
                    CK(ctx, cudaStreamWaitEvent(ks, d.ev_rout[si], 0));   // the scratch's last outputs have left
                    if (any_pageable) CK(ctx, cudaEventSynchronize(d.ev_rin[si]));   // so has the staging's last input
                    size_t off = 0;
                    for (int b = 0; b < n_in; b++) {
                        const size_t w = in_words(b, cnt);
                        if (in_pageable[b]) memcpy(d.ray_stage[si] + off, src[b], w * sizeof(float));
                        CK(ctx, cudaMemcpyAsync(d.ray_mem[si] + off, in_pageable[b] ? d.ray_stage[si] + off : src[b],
                                                w * sizeof(float), cudaMemcpyHostToDevice, ks));
                        src[b] = d.ray_mem[si] + off;
                        off += w;
                    }
                    CK(ctx, cudaEventRecord(d.ev_rin[si], ks));
                    // every output goes to the scratch; only the requested ones leave it
                    for (int b = 0; b < n_out; b++) dst[b] = out_dev(si, cnt, b);
                } else {
                    for (int b = 0; b < n_out; b++)
                        if (out[b]) dst[b] = out[b] + a * out_bytes[b];
                }
                unsigned char* ctl = d.ray_ctl + 64 * si;
                CK(ctx, cudaMemsetAsync(ctl, 0, sizeof(unsigned int), ks));
                RenderLaunch rl = band_launch(ctx, d, p, 0, 0, occ ? nullptr : static_cast<float*>(dst[0]),
                                              reinterpret_cast<unsigned int*>(ctl));
                rl.counters = reinterpret_cast<unsigned long long*>(ctl + 8);
                rl.ray_invalid = reinterpret_cast<unsigned long long*>(ctl + 32);
                rl.list_n = (int)cnt;
                if (!points) {
                    rl.ray_o = src[1];
                    rl.ray_o_stride = shared_origin ? 0 : 3;
                    rl.ray_d = src[0];
                }
                if (occ) {
                    OccLaunch ol{};
                    ol.rl = rl;
                    ol.tmax = points ? nullptr : src[2];
                    ol.points = points ? src[0] : nullptr;
                    ol.out = static_cast<unsigned char*>(dst[0]);
                    CK(ctx, tcrt_launch_occlusion(ol, d.sm_count, ks));
                } else if (views) {
                    // pixel (xc, z) of the piece is global column a + xc
                    rl.x0 = (int)a;
                    rl.x1 = (int)(a + cnt);
                    rl.out = dst[0] ? static_cast<float*>(dst[0]) : d.ray_mem[si];
                    rl.view_cams = d.view_cams;
                    CK(ctx, tcrt_launch_render_views(rl, d.sm_count, ks));
                    if (out[1]) {
                        CK(ctx, tcrt_launch_quantize8(rl.out, cnt * col_px, static_cast<unsigned char*>(dst[1]), ks));
                        launches[i]++;
                    }
                } else if (hits) {
                    HitLaunch hl{};
                    hl.rl = rl;
                    hl.object = static_cast<int*>(dst[0]);
                    hl.distance = static_cast<float*>(dst[1]);
                    hl.normal = static_cast<float*>(dst[2]);
                    CK(ctx, tcrt_launch_hits(hl, d.sm_count, ks));
                } else {
                    CK(ctx, tcrt_launch_render_rays(rl, d.sm_count, ks));
                }
                launches[i]++;
                CK(ctx, cudaEventRecord(d.ev_rk[si], ks));
            }
            if (!device_form && k >= lag && (rc = send_out(k - lag))) return rc;
        }
        for (int si = 1; si < ns; si++) CK(ctx, cudaStreamWaitEvent(d.stream, d.ev_rk[si], 0));
        CK(ctx, cudaEventRecord(d.ev_r1, d.stream));
        CK(ctx, cudaMemcpyAsync(d.h_ray, d.ray_ctl, 64 * ns, cudaMemcpyDeviceToHost, d.stream));
        if (!device_form) CK(ctx, cudaEventRecord(d.ev_rc, d.copy_stream));
    }
    unsigned long long bad = 0, n_launches = 0;
    for (int i = d_begin; i < d_end; i++) {
        DeviceState& d = ctx->devs[i];
        if (stats) {
            stats->col_begin[i] = (int)std::min<size_t>(cut[i], INT_MAX);
            stats->col_end[i] = (int)std::min<size_t>(cut[i + 1], INT_MAX);
        }
        if (used_streams[i] == 0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));
        if (!device_form) CK(ctx, cudaEventSynchronize(d.ev_rc));
        unsigned long long cnt[4] = {0, 0, 0, 0};   // primary, shadow, reflect, invalid
        for (int si = 0; si < used_streams[i]; si++)
            for (int c = 0; c < 4; c++) cnt[c] += d.h_ray[8 * si + 1 + c];
        if (hits) cnt[0] = (cut[i + 1] - cut[i]) - cnt[3];
        bad += cnt[3];
        n_launches += (unsigned long long)launches[i];
        if (stats) {
            float ms = 0.f;
            CK(ctx, cudaEventElapsedTime(&ms, d.ev_r0, d.ev_r1));
            stats->render_ms[i] = ms;
            if (!device_form) {
                CK(ctx, cudaEventElapsedTime(&ms, d.ev_r1, d.ev_rc));
                stats->d2h_ms[i] = std::max(ms, 0.f);   // copy time not hidden behind the kernels
            }
            stats->rays_primary[i] = cnt[0];
            stats->rays_shadow[i] = cnt[1];
            stats->rays_reflect[i] = cnt[2];
        }
    }
    if (stats) {
        stats->n_devices = nd;
        stats->gpu_launches = n_launches;
    }
    if (n_invalid) *n_invalid = bad;
    return TCRT_OK;
}

extern "C" {

int tcrt_trace_rays(tcrt_ctx* ctx, const tcrt_params* p, size_t n, const float* origins, int shared_origin,
                    const float* directions, float* rgb, unsigned long long* n_invalid, tcrt_stats* stats) {
    void* out[3] = {rgb, nullptr, nullptr};
    return rays_impl(ctx, -1, kBatchColour, p, n, origins, shared_origin, directions, nullptr, out, n_invalid, stats);
}

int tcrt_intersect_rays(tcrt_ctx* ctx, const tcrt_params* p, size_t n, const float* origins, int shared_origin,
                        const float* directions, int* object, float* distance, float* normal,
                        unsigned long long* n_invalid, tcrt_stats* stats) {
    void* out[3] = {object, distance, normal};
    return rays_impl(ctx, -1, kBatchHits, p, n, origins, shared_origin, directions, nullptr, out, n_invalid, stats);
}

int tcrt_trace_rays_device(tcrt_ctx* ctx, int device_slot, const tcrt_params* p, size_t n, const float* origins,
                           int shared_origin, const float* directions, float* rgb, unsigned long long* n_invalid,
                           tcrt_stats* stats) {
    if (device_slot < 0) return fail(ctx, TCRT_ERR_INVALID, "device slot %d out of range", device_slot);
    void* out[3] = {rgb, nullptr, nullptr};
    return rays_impl(ctx, device_slot, kBatchColour, p, n, origins, shared_origin, directions, nullptr, out, n_invalid, stats);
}

int tcrt_intersect_rays_device(tcrt_ctx* ctx, int device_slot, const tcrt_params* p, size_t n, const float* origins,
                               int shared_origin, const float* directions, int* object, float* distance, float* normal,
                               unsigned long long* n_invalid, tcrt_stats* stats) {
    if (device_slot < 0) return fail(ctx, TCRT_ERR_INVALID, "device slot %d out of range", device_slot);
    void* out[3] = {object, distance, normal};
    return rays_impl(ctx, device_slot, kBatchHits, p, n, origins, shared_origin, directions, nullptr, out, n_invalid, stats);
}

int tcrt_occluded_rays(tcrt_ctx* ctx, size_t n, const float* origins, int shared_origin, const float* directions,
                       const float* tmax, unsigned char* occluded, unsigned long long* n_invalid, tcrt_stats* stats) {
    void* out[3] = {occluded, nullptr, nullptr};
    return rays_impl(ctx, -1, kBatchOccRays, nullptr, n, origins, shared_origin, directions, tmax, out, n_invalid, stats);
}

int tcrt_occluded_lights(tcrt_ctx* ctx, size_t n, const float* points, unsigned char* occluded,
                         unsigned long long* n_invalid, tcrt_stats* stats) {
    void* out[3] = {occluded, nullptr, nullptr};
    return rays_impl(ctx, -1, kBatchOccPoints, nullptr, n, nullptr, 0, points, nullptr, out, n_invalid, stats);
}

int tcrt_occluded_rays_device(tcrt_ctx* ctx, int device_slot, size_t n, const float* origins, int shared_origin,
                              const float* directions, const float* tmax, unsigned char* occluded,
                              unsigned long long* n_invalid, tcrt_stats* stats) {
    if (device_slot < 0) return fail(ctx, TCRT_ERR_INVALID, "device slot %d out of range", device_slot);
    void* out[3] = {occluded, nullptr, nullptr};
    return rays_impl(ctx, device_slot, kBatchOccRays, nullptr, n, origins, shared_origin, directions, tmax, out, n_invalid,
                     stats);
}

int tcrt_occluded_lights_device(tcrt_ctx* ctx, int device_slot, size_t n, const float* points, unsigned char* occluded,
                                unsigned long long* n_invalid, tcrt_stats* stats) {
    if (device_slot < 0) return fail(ctx, TCRT_ERR_INVALID, "device slot %d out of range", device_slot);
    void* out[3] = {occluded, nullptr, nullptr};
    return rays_impl(ctx, device_slot, kBatchOccPoints, nullptr, n, nullptr, 0, points, nullptr, out, n_invalid, stats);
}

}  // extern "C"

// Multi-view frames: the n_views * width global columns of the stacked views as a batch of kind kBatchViews.
static int views_impl(tcrt_ctx* ctx, int slot, const tcrt_params* p, int n_views, const tcrt_camera* cams, float* rgb,
                      unsigned char* rgb8, tcrt_stats* stats) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null ctx");
    if (!p) return fail(ctx, TCRT_ERR_INVALID, "null params");
    if (n_views < 0) return fail(ctx, TCRT_ERR_INVALID, "n_views %d < 0", n_views);
    if (!valid_params(p)) return fail(ctx, TCRT_ERR_INVALID, "bad params");
    if ((long long)n_views * p->width > INT_MAX)
        return fail(ctx, TCRT_ERR_UNSUPPORTED, "%d views of width %d: more than INT_MAX columns", n_views, p->width);
    void* out[3] = {rgb, rgb8, nullptr};
    return rays_impl(ctx, slot, kBatchViews, p, (size_t)n_views * (size_t)p->width, nullptr, 0, nullptr, nullptr, out,
                     nullptr, stats, cams);
}

extern "C" {

int tcrt_render_views(tcrt_ctx* ctx, const tcrt_params* p, int n_views, const tcrt_camera* cameras, float* rgb,
                      unsigned char* rgb8, tcrt_stats* stats) {
    return views_impl(ctx, -1, p, n_views, cameras, rgb, rgb8, stats);
}

int tcrt_render_views_device(tcrt_ctx* ctx, int device_slot, const tcrt_params* p, int n_views, const tcrt_camera* cameras,
                             float* rgb, unsigned char* rgb8, tcrt_stats* stats) {
    if (device_slot < 0) return fail(ctx, TCRT_ERR_INVALID, "device slot %d out of range", device_slot);
    return views_impl(ctx, device_slot, p, n_views, cameras, rgb, rgb8, stats);
}

}  // extern "C"

// ---- adaptive frames (tcrt_adaptive.cu): supersample only the pixels at contrast edges ------------------------------------
// Samples traced per piece of the refined list: 4 M samples = 48 MB of sample scratch per render stream, far inside the
// kernels' int index range at every ss.
constexpr long long kPieceSamples = 1LL << 22;

// Per device band [bx0, bx1) (equal widths; the balancer's cut and cost map are neither read nor updated):
//   1. the plain frame over [bx0 - 1, bx1 + 1) clipped to the frame, column chunks round robin over the render streams;
//   2. classify + scan + compact on the render stream: mask, the plain pixels copied into the band's frame, the list;
//   3. the list's length to the host (it sizes step 4): one 4-byte copy and a wait;
//   4. pieces of the list round robin over the render streams, each one list-mode render launch of samples 1 .. ss*ss-1
//      into the stream's sample scratch and one resolve launch into the frame;
//   5. RGB8: one quantisation launch over the band; then the band and the mask to the host.
// Steps 1-2 run on all devices before any waits in step 3, and step 4 on all before any waits in step 5.
static int render_adaptive(tcrt_ctx* ctx, const tcrt_params* p, int ss, int contrast, int x0, int x1, void* host_band,
                           FrameFormat fmt, unsigned char* host_mask, unsigned long long* n_refined, tcrt_stats* stats) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null ctx");
    if (ss < 1) return fail(ctx, TCRT_ERR_INVALID, "samples per axis %d < 1", ss);
    if (contrast < -1 || contrast > 255) return fail(ctx, TCRT_ERR_INVALID, "contrast %d outside [-1, 255]", contrast);
    int rc = check_ss(ctx, p, ss);
    if (rc) return rc;
    if (!valid_params(p)) return fail(ctx, TCRT_ERR_INVALID, "bad params");
    if (x0 < 0 || x1 > p->width || x0 >= x1) return fail(ctx, TCRT_ERR_INVALID, "bad column range [%d,%d)", x0, x1);
    if (p->max_depth > TCRT_MAX_DEPTH)
        return fail(ctx, TCRT_ERR_UNSUPPORTED, "max_depth %d > TCRT_MAX_DEPTH %d", p->max_depth, TCRT_MAX_DEPTH);
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    const int set = ctx->devs[0].cur;
    if (ctx->pend[set].active)
        return fail(ctx, TCRT_ERR_INVALID, "a frame submitted with tcrt_render_async is still pending in this slot: tcrt_wait first");
    const int nd = (int)ctx->devs.size();
    const int W = p->width, H = p->height;
    const int m = ss * ss - 1;                           // samples traced per refined pixel
    tcrt_params sp = *p;                                 // the sample frame the list-mode launches trace
    sp.width = ss * W;
    sp.height = ss * H;
    std::vector<int> cut(nd + 1);
    for (int i = 0; i <= nd; i++) cut[i] = x0 + (int)((long long)(x1 - x0) * i / nd);
    // pageable destinations of at least 512 K pixels go through the pinned staging, as frames do (render_impl)
    const bool big = (long long)(x1 - x0) * H >= 512 * 1024;
    const bool staged_frame = host_band && big && host_pageable(host_band);
    const bool staged_mask = host_mask && big && host_pageable(host_mask);
    const bool any_direct = (host_band && !staged_frame) || (host_mask && !staged_mask);
    const size_t bpp = bytes_per_px(fmt);
    ctx->has_frame = false;
    ctx->txt_prepared = false;
    int launches = 0;
    auto queue_of = [](DeviceState& d, int si) { return reinterpret_cast<unsigned int*>(d.fr().ctl + 64) + si; };
    auto stream_of = [](DeviceState& d, int si) { return si == 0 ? d.stream : d.chunk_stream[si - 1]; };
    // the render streams 1.. join the render stream: ev_chunk[si] marks stream si's last launch
    auto join = [&](DeviceState& d, int n_streams) -> int {
        for (int si = 1; si < n_streams; si++) {
            CK(ctx, cudaEventRecord(d.fr().ev_chunk[si], stream_of(d, si)));
            CK(ctx, cudaStreamWaitEvent(d.stream, d.fr().ev_chunk[si], 0));
        }
        return TCRT_OK;
    };
    // ...and wait for what the render stream has queued so far (ev_start)
    auto fork = [&](DeviceState& d, int n_streams) -> int {
        CK(ctx, cudaEventRecord(d.fr().ev_start, d.stream));
        for (int si = 1; si < n_streams; si++) CK(ctx, cudaStreamWaitEvent(stream_of(d, si), d.fr().ev_start, 0));
        return TCRT_OK;
    };
    // ---- 1-2: plain pass and classification ----------------------------------------------------------------------------------
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        FrameRes& f = d.fr();
        f.x0 = cut[i];
        f.x1 = cut[i + 1];
        f.height = H;
        f.n_chunks = 0;      // the band has no chunk events: the whole band is complete when the call returns
        if (f.x1 <= f.x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        const int bx0 = f.x0, bx1 = f.x1, hx0 = std::max(0, bx0 - 1), hx1 = std::min(W, bx1 + 1);
        const size_t n_px = (size_t)(bx1 - bx0) * H;
        const size_t nb = (n_px + 255) / 256;
        rc = ensure(ctx, f.frame, f.frame_cap, 3 * n_px);
        if (!rc && fmt == kRGB8) rc = ensure(ctx, f.frame8, f.frame8_cap, 3 * n_px);
        if (!rc) rc = ensure(ctx, d.ad_plain, d.ad_plain_cap, (size_t)(hx1 - hx0) * H * 3);
        if (!rc) rc = ensure(ctx, d.ad_mask, d.ad_mask_cap, n_px);
        if (!rc) rc = ensure(ctx, d.ad_counts, d.ad_counts_cap, nb + 1);
        if (!rc) rc = ensure(ctx, d.ad_list, d.ad_list_cap, n_px);
        if (rc) return rc;
        CK(ctx, cudaMemsetAsync(f.ctl, 0, 64 + kMaxChunks * sizeof(unsigned int), d.stream));
        CK(ctx, cudaEventRecord(f.ev_k0, d.stream));
        // column chunks of the halo band as plain frames are chunked (plan_chunks)
        FrameRes plan;
        plan.x0 = hx0;
        plan.x1 = hx1;
        plan_chunks(plan, H, true);
        const int n_streams = ctx->one_stream ? 1 : std::min(kChunkStreams, plan.n_chunks);
        rc = fork(d, n_streams);
        if (rc) return rc;
        for (int k = 0; k < plan.n_chunks; k++) {
            const int cx0 = plan.chunk_x[k], cx1 = plan.chunk_x[k + 1];
            if (cx1 <= cx0) continue;
            const int si = k % n_streams;
            const cudaStream_t ks = stream_of(d, si);
            CK(ctx, cudaMemsetAsync(queue_of(d, si), 0, sizeof(unsigned int), ks));
            const RenderLaunch rl = band_launch(ctx, d, p, cx0, cx1, d.ad_plain + (size_t)(cx0 - hx0) * H * 3, queue_of(d, si));
            CK(ctx, tcrt_launch_render(rl, d.sm_count, ks, &launches, nullptr, 0));
        }
        rc = join(d, n_streams);
        if (rc) return rc;
        CK(ctx, tcrt_launch_adaptive_classify(d.ad_plain, hx0, W, H, bx0, bx1, contrast, f.frame, d.ad_mask, d.ad_counts,
                                              d.ad_list, d.stream));
        launches += 3;
        f.h_counters[0] = 0;     // slot 0 of the counters is free: the list's length goes there
        CK(ctx, cudaMemcpyAsync(f.h_counters, d.ad_counts + nb, sizeof(unsigned int), cudaMemcpyDeviceToHost, d.stream));
        CK(ctx, cudaEventRecord(f.ev_done, d.stream));
    }
    // ---- 3: the lists' lengths -------------------------------------------------------------------------------------------------
    std::vector<long long> n_list(nd, 0);
    unsigned long long total = 0;
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        if (d.fr().x1 <= d.fr().x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaEventSynchronize(d.fr().ev_done));
        n_list[i] = (long long)(d.fr().h_counters[0] & 0xffffffffull);
        total += (unsigned long long)n_list[i];
    }
    // ---- 4: sample pass --------------------------------------------------------------------------------------------------------
    const long long per_piece = std::max(1LL, kPieceSamples / std::max(1, m));    // list entries per piece
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        FrameRes& f = d.fr();
        if (f.x1 <= f.x0 || ss == 1 || n_list[i] == 0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        const int n_pieces = (int)((n_list[i] + per_piece - 1) / per_piece);
        const int n_streams = ctx->one_stream ? 1 : std::min(kChunkStreams, n_pieces);
        const size_t need = (size_t)std::min(n_list[i], per_piece) * m * 3;
        for (int si = 0; si < n_streams; si++)     // a buffer about to be replaced may still serve a frame in flight
            if (need > d.ss_scratch_cap[si]) {
                CK(ctx, cudaDeviceSynchronize());
                break;
            }
        for (int si = 0; si < n_streams; si++) {
            rc = ensure(ctx, d.ss_scratch[si], d.ss_scratch_cap[si], need);
            if (rc) return rc;
        }
        rc = fork(d, n_streams);
        if (rc) return rc;
        for (int k = 0; k < n_pieces; k++) {
            const long long e0 = (long long)k * per_piece, cnt = std::min(per_piece, n_list[i] - e0);
            const int si = k % n_streams;
            const cudaStream_t ks = stream_of(d, si);
            CK(ctx, cudaMemsetAsync(queue_of(d, si), 0, sizeof(unsigned int), ks));
            RenderLaunch rl = band_launch(ctx, d, &sp, 0, sp.width, d.ss_scratch[si], queue_of(d, si));
            rl.list = d.ad_list + e0;
            rl.list_n = (int)(cnt * m);
            rl.list_ss = ss;
            CK(ctx, tcrt_launch_render_list(rl, d.sm_count, ks));
            CK(ctx, tcrt_launch_adaptive_resolve(d.ad_list, (int)e0, (int)cnt, f.x0, H, ss, d.ss_scratch[si], f.frame, ks));
            launches += 2;
        }
        rc = join(d, n_streams);
        if (rc) return rc;
    }
    // ---- 5: output -------------------------------------------------------------------------------------------------------------
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        FrameRes& f = d.fr();
        if (f.x1 <= f.x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        const size_t n_px = (size_t)(f.x1 - f.x0) * H;
        if (fmt == kRGB8) {
            CK(ctx, tcrt_launch_quantize8(f.frame, n_px, f.frame8, d.stream));
            launches++;
        }
        CK(ctx, cudaEventRecord(f.ev_k1, d.stream));
        CK(ctx, cudaMemcpyAsync(f.h_counters, f.ctl, 32, cudaMemcpyDeviceToHost, d.stream));
        CK(ctx, cudaEventRecord(f.ev_done, d.stream));
        if (any_direct) {
            CK(ctx, cudaStreamWaitEvent(d.copy_stream, f.ev_k1, 0));
            if (host_band && !staged_frame)
                CK(ctx, cudaMemcpyAsync(static_cast<char*>(host_band) + (size_t)(f.x0 - x0) * H * bpp, frame_src(f, fmt),
                                        n_px * bpp, cudaMemcpyDeviceToHost, d.copy_stream));
            if (host_mask && !staged_mask)
                CK(ctx, cudaMemcpyAsync(host_mask + (size_t)(f.x0 - x0) * H, d.ad_mask, n_px, cudaMemcpyDeviceToHost,
                                        d.copy_stream));
            CK(ctx, cudaEventRecord(f.ev_c1, d.copy_stream));
        }
    }
    // pageable destinations: through the pinned staging slots and the copy workers, band after band
    for (int k = 0; k < 2; k++) {
        if (!(k == 0 ? staged_frame : staged_mask)) continue;
        const size_t b = k == 0 ? bpp : 1;
        TxtPipe& pipe = copy_pipe_to(ctx, k == 0 ? host_band : host_mask);
        cudaError_t e = cudaSuccess;
        for (auto& d : ctx->devs) {
            FrameRes& f = d.fr();
            if (f.x1 <= f.x0) continue;
            const char* src = k == 0 ? frame_src(f, fmt) : reinterpret_cast<const char*>(d.ad_mask);
            e = cudaSetDevice(d.dev);
            if (e == cudaSuccess) e = ensure_stage(d);
            StageSlots slots;
            if (e == cudaSuccess) e = stage_out(pipe, d, slots, src, (size_t)(f.x1 - f.x0) * H * b, (size_t)(f.x0 - x0) * H * b, f.ev_k1);
            slots.drain(pipe);
            if (e != cudaSuccess) break;
        }
        if (e != cudaSuccess || pipe.io_error)
            return fail(ctx, TCRT_ERR_CUDA, "staged copy-out of an adaptive %s: %s", k == 0 ? "frame" : "mask",
                        e != cudaSuccess ? cudaGetErrorString(e) : "a chunk did not arrive");
    }
    if (stats) memset(stats, 0, sizeof(*stats));
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        FrameRes& f = d.fr();
        if (stats) {
            stats->col_begin[i] = f.x0;
            stats->col_end[i] = f.x1;
        }
        if (f.x1 <= f.x0) continue;
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaEventSynchronize(f.ev_done));
        if (any_direct) CK(ctx, cudaEventSynchronize(f.ev_c1));
        if (stats) {
            float ms = 0.f;
            CK(ctx, cudaEventElapsedTime(&ms, f.ev_k0, f.ev_k1));
            stats->render_ms[i] = ms;
            if (any_direct) CK(ctx, cudaEventElapsedTime(&ms, f.ev_k1, f.ev_c1));
            stats->d2h_ms[i] = any_direct ? std::max(ms, 0.f) : 0.0;
            stats->rays_primary[i] = f.h_counters[1];
            stats->rays_shadow[i] = f.h_counters[2];
            stats->rays_reflect[i] = f.h_counters[3];
        }
    }
    if (stats) {
        stats->n_devices = nd;
        stats->gpu_launches = (unsigned long long)launches;
    }
    if (n_refined) *n_refined = total;
    ctx->has_frame = true;
    ctx->txt_prepared = false;
    ctx->frame_x0 = x0;
    ctx->frame_x1 = x1;
    ctx->frame_h = H;
    return TCRT_OK;
}

extern "C" {

int tcrt_render_columns_adaptive(tcrt_ctx* ctx, const tcrt_params* p, int ss, int contrast, int x0, int x1, float* host_rgb_band,
                                 unsigned char* host_mask, unsigned long long* n_refined, tcrt_stats* stats) {
    return render_adaptive(ctx, p, ss, contrast, x0, x1, host_rgb_band, kFloat32, host_mask, n_refined, stats);
}

int tcrt_render_columns_adaptive_rgb8(tcrt_ctx* ctx, const tcrt_params* p, int ss, int contrast, int x0, int x1,
                                      unsigned char* host_rgb8_band, unsigned char* host_mask, unsigned long long* n_refined,
                                      tcrt_stats* stats) {
    if (!host_rgb8_band) return fail(ctx, TCRT_ERR_INVALID, "null output buffer");
    return render_adaptive(ctx, p, ss, contrast, x0, x1, host_rgb8_band, kRGB8, host_mask, n_refined, stats);
}

}  // extern "C"

namespace {

// A mapping pays on memory-backed files (tmpfs, where the page cache IS the file: measured 45 ms against 76 ms
// for a 4K frame); on a disk-backed file system dirtying mapped pages is slower than pwrite (measured 2-5x).
void map_sink(TxtSink* s) {
    struct statfs fs;
    const bool memory_backed = fstatfs(s->fd, &fs) == 0 && (fs.f_type == 0x01021994 /* TMPFS_MAGIC */ || fs.f_type == 0x858458f6 /* RAMFS_MAGIC */);
    if (!memory_backed) return;
    void* m = mmap(nullptr, s->size, PROT_READ | PROT_WRITE, MAP_SHARED, s->fd, 0);
    s->map = (m == MAP_FAILED) ? nullptr : static_cast<char*>(m);
}

// Opens (create or keep) the file, sizes it when `size` != 0, maps it for writing when that pays; else pwrite.
int open_sink(tcrt_ctx* ctx, const char* path, bool create, size_t size, TxtSink* s) {
    s->fd = open(path, create ? (O_RDWR | O_CREAT | O_TRUNC) : O_RDWR, 0666);
    if (s->fd < 0) return fail(ctx, TCRT_ERR_IO, "Error Opening File %s", path);
    if (create && size && ftruncate(s->fd, (off_t)size) != 0) {
        close(s->fd);
        s->fd = -1;
        return fail(ctx, TCRT_ERR_IO, "cannot size %s to %zu bytes", path, size);
    }
    s->size = size;
    if (size) map_sink(s);
    return TCRT_OK;
}

bool close_sink(TxtSink* s, size_t final_size) {
    bool ok = true;
    if (s->map) ok = munmap(s->map, s->size) == 0 && ok;
    s->map = nullptr;
    if (s->fd >= 0) {
        if (final_size != s->size) ok = ftruncate(s->fd, (off_t)final_size) == 0 && ok;
        ok = close(s->fd) == 0 && ok;
    }
    s->fd = -1;
    return ok;
}

}  // namespace

extern "C" {

// Streams every device's band through the pipe (one issuing thread per device, the caller's thread for device 0).
// Exceptions of the C++ runtime (thread creation) must not cross the C boundary: they become TCRT_ERR_IO.
static int stream_all_bands(tcrt_ctx* ctx, const TxtSink& sink, size_t base, bool* any_not_fixed, bool* io_error) {
    const int nd = (int)ctx->devs.size();
    std::vector<int> rcs(nd, TCRT_OK);
    std::vector<unsigned int> not_fixed(nd, 0u);
    std::vector<std::string> errs(nd);
    TxtPipe pipe;
    std::vector<std::thread> issuers;
    try {
        pipe.start(&sink, n_txt_workers());
        for (int i = 1; i < nd; i++)
            issuers.emplace_back([&, i] { rcs[i] = stream_band_fixed(ctx, ctx->devs[i], pipe, base, &not_fixed[i], &errs[i]); });
        rcs[0] = stream_band_fixed(ctx, ctx->devs[0], pipe, base, &not_fixed[0], &errs[0]);
        for (auto& t : issuers) t.join();
        pipe.finish();
    } catch (const std::exception& e) {
        for (auto& t : issuers)
            if (t.joinable()) t.join();
        pipe.finish();
        return fail(ctx, TCRT_ERR_IO, "writer threads: %s", e.what());
    }
    ctx->txt_prepared = false;
    *any_not_fixed = false;
    *io_error = pipe.io_error;
    for (int i = 0; i < nd; i++) {
        if (rcs[i]) return fail(ctx, rcs[i], "%s", errs[i].c_str());
        *any_not_fixed = *any_not_fixed || not_fixed[i] != 0u;
    }
    return TCRT_OK;
}

// General layout (some line is not 31 bytes): per-pixel lengths -> scan -> byte stores, whole bands at a time.
static int write_txt_general(tcrt_ctx* ctx, const char* path, const char* header, int hn) {
    size_t total = 0;
    int rc = tcrt_txt_size(ctx, &total);
    if (rc) return rc;
    if (total + 16 > ctx->host_text_cap) {
        if (ctx->host_text) cudaFreeHost(ctx->host_text);
        ctx->host_text = nullptr;
        ctx->host_text_cap = 0;
        CK(ctx, cudaHostAlloc((void**)&ctx->host_text, total + 16, cudaHostAllocPortable));
        ctx->host_text_cap = total + 16;
    }
    rc = tcrt_format_txt(ctx, ctx->host_text, ctx->host_text_cap, &total);
    if (rc) return rc;
    // fopen(path, "w") semantics (log_file_mode "w", RayTracer.h:135): create or truncate
    int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC, 0666);
    if (fd < 0) return fail(ctx, TCRT_ERR_IO, "Error Opening File %s", path);
    bool ok = write_fully(fd, header, (size_t)hn) && write_fully(fd, ctx->host_text, total);
    ok = (close(fd) == 0) && ok;
    if (!ok) return fail(ctx, TCRT_ERR_IO, "short write to %s", path);
    return TCRT_OK;
}

int tcrt_write_txt(tcrt_ctx* ctx, const tcrt_params* p, const char* path, double run_time_s) {
    if (!ctx || !p || !path) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    int rc = check_full_frame(ctx, p);
    if (rc) return rc;
    char header[512];
    const int hn = tcrt_txt_header(p, run_time_s, header, sizeof header);
    if (hn < 0) return fail(ctx, TCRT_ERR_INVALID, "header formatting failed");
    // fixed-width attempt: header + W*H lines of 31 bytes, every band streamed by its own issuing thread
    const size_t total = (size_t)hn + (size_t)p->width * p->height * kTxtLine;
    TxtSink sink;
    rc = open_sink(ctx, path, true, total, &sink);
    if (rc) return rc;
    sink.put(0, header, (size_t)hn);
    bool general = false, io_error = false;
    rc = stream_all_bands(ctx, sink, (size_t)hn, &general, &io_error);
    if (rc) {
        close_sink(&sink, total);
        return rc;
    }
    if (!close_sink(&sink, total) || io_error) return fail(ctx, TCRT_ERR_IO, "short write to %s", path);
    if (general) return write_txt_general(ctx, path, header, hn);
    return TCRT_OK;
}

int tcrt_txt_create(const tcrt_params* p, const char* path, double run_time_s) {
    if (!p || !path || !valid_params(p)) return fail(nullptr, TCRT_ERR_INVALID, "bad argument");
    char header[512];
    const int hn = tcrt_txt_header(p, run_time_s, header, sizeof header);
    if (hn < 0) return fail(nullptr, TCRT_ERR_INVALID, "header formatting failed");
    int fd = open(path, O_RDWR | O_CREAT | O_TRUNC, 0666);
    if (fd < 0) return fail(nullptr, TCRT_ERR_IO, "Error Opening File %s", path);
    bool ok = ftruncate(fd, (off_t)((size_t)hn + (size_t)p->width * p->height * kTxtLine)) == 0 && write_fully(fd, header, (size_t)hn);
    ok = (close(fd) == 0) && ok;
    if (!ok) return fail(nullptr, TCRT_ERR_IO, "cannot create %s", path);
    return TCRT_OK;
}

int tcrt_write_txt_band(tcrt_ctx* ctx, const tcrt_params* p, const char* path, double run_time_s) {
    if (!ctx || !p || !path) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (!ctx->has_frame) return fail(ctx, TCRT_ERR_NO_FRAME, "nothing rendered yet");
    if (ctx->frame_h != p->height || ctx->frame_x1 > p->width)
        return fail(ctx, TCRT_ERR_INVALID, "last render does not belong to a %dx%d image", p->width, p->height);
    char header[512];
    const int hn = tcrt_txt_header(p, run_time_s, header, sizeof header);
    if (hn < 0) return fail(ctx, TCRT_ERR_INVALID, "header formatting failed");
    const size_t total = (size_t)hn + (size_t)p->width * p->height * kTxtLine;
    TxtSink sink;
    int rc = open_sink(ctx, path, false, 0, &sink);
    if (rc) return rc;
    struct stat st;
    if (fstat(sink.fd, &st) != 0 || (size_t)st.st_size != total) {
        close_sink(&sink, 0);
        return fail(ctx, TCRT_ERR_INVALID, "%s was not made by tcrt_txt_create for these params", path);
    }
    sink.size = total;
    map_sink(&sink);
    bool not_fixed = false, io_error = false;
    rc = stream_all_bands(ctx, sink, (size_t)hn, &not_fixed, &io_error);
    const bool closed = close_sink(&sink, total);
    if (rc) return rc;
    if (not_fixed)
        return fail(ctx, TCRT_ERR_UNSUPPORTED, "a pixel line of this band is not 31 bytes (a channel >= 10, negative or not finite): "
                                               "gather the bands and use tcrt_write_txt");
    if (!closed || io_error) return fail(ctx, TCRT_ERR_IO, "short write to %s", path);
    return TCRT_OK;
}

}  // extern "C"

// ---- moving spheres (tcrt_update_spheres) ------------------------------------------------------------------------------------
// The spheres of the resident scene take new centres and radii on every device, in place: tcrt_update.cu scatters them into
// the blob, refits the sphere BVH and re-registers the sphere grid; the host then recomputes what the launches take by
// value (scene_scalars) and the light rows (light_rows) from one small read-back, with the upload's own code.  Planes,
// materials, textures and counts stay.  DESIGN.md §4.3, §4.5.

// bytes of device memory from `off` on, rounded so that the next piece starts 256-byte aligned
static size_t carve(size_t& off, size_t bytes) {
    const size_t at = off;
    off += (bytes + 255) & ~(size_t)255;
    return at;
}

// ctx->upd_stage with room for `f4` float4s
static int ensure_upd_stage(tcrt_ctx* ctx, size_t f4) {
    if (f4 <= ctx->upd_stage_cap) return TCRT_OK;
    if (ctx->upd_stage) cudaFreeHost(ctx->upd_stage);
    ctx->upd_stage = nullptr;
    ctx->upd_stage_cap = 0;
    CK(ctx, cudaHostAlloc((void**)&ctx->upd_stage, f4 * sizeof(float4), cudaHostAllocPortable));
    ctx->upd_stage_cap = f4;
    return TCRT_OK;
}

// What the sphere launches leave for the host: the spheres' part of the bounds, whether the grid stays, the max |centre
// component| they reduced, the lights' positions, and per device the grid's item list and the launches' device time.
struct SpherePass {
    SceneBounds bounds;
    bool keep_grid = false;
    double ext_sph = 0.0;
    std::vector<float> og;
    std::vector<int*> items;
    std::vector<float> ms;
    bool invalid = false;        // a resident sphere is not finite (a rebox): nothing was written
};

// The sphere update's launches on every device, after the frames queued before the call, and their read-back.  rebox: the
// resident spheres stay where they are and are boxed again with the ext of ext_fixed (a plane update that raised it); geom
// is then unused.  Nothing of the scene changes when the input is invalid.
static int sphere_pass(tcrt_ctx* ctx, int slot, const float* geom, bool rebox, double ext_fixed, SpherePass& out,
                       int* launches) {
    const int nd = (int)ctx->devs.size();
    const int src_dev = slot >= 0 ? ctx->devs[slot].dev : -1;
    const UpdatePlan& up = ctx->scene_upd;
    const int n = up.n_spheres;
    const DeviceScene& ds0 = ctx->scene_ds;
    const bool grid = ctx->scene_grid;
    const int n_bvh = ds0.n_sph_bvh, n_ls = (int)up.light_sph.size(), n_levels = (int)up.level_start.size() - 1;
    const unsigned cap = 8u * (unsigned)n_bvh;
    const size_t back_bytes = sizeof(UpdateBack) + 12 * (size_t)n_ls;
    if (int rc = ensure_upd_stage(ctx, std::max((size_t)n, 2 * (size_t)ds0.n_lights))) return rc;
    if (slot < 0 && !rebox) memcpy(ctx->upd_stage, geom, (size_t)n * sizeof(float4));
    out.items.assign(nd, nullptr);
    out.ms.assign(nd, 0.f);
    // the maps: slot_of, light_sph, levels, level_start, then for a rebox the identity and the light spheres' slots
    const size_t o_ident = (size_t)n + n_ls + up.levels.size() + up.level_start.size();
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));   // frames queued before the call finish with the old scene
        if (!d.ev_u0) CK(ctx, cudaEventCreate(&d.ev_u0));
        if (!d.ev_u1) CK(ctx, cudaEventCreate(&d.ev_u1));
        // the upload's maps, once per upload
        const size_t n_maps = o_ident + (size_t)n + n_ls;
        int rc = ensure(ctx, d.upd_maps, d.upd_maps_cap, n_maps);
        if (rc) return rc;
        if (d.upd_serial != ctx->scene_serial) {
            std::vector<int> maps(up.slot_of);
            maps.insert(maps.end(), up.light_sph.begin(), up.light_sph.end());
            maps.insert(maps.end(), up.levels.begin(), up.levels.end());
            maps.insert(maps.end(), up.level_start.begin(), up.level_start.end());
            for (int k = 0; k < n; k++) maps.push_back(k);
            for (int j = 0; j < n_ls; j++) maps.push_back(up.slot_of[up.light_sph[j]]);
            CK(ctx, cudaMemcpy(d.upd_maps, maps.data(), maps.size() * sizeof(int), cudaMemcpyHostToDevice));
            d.upd_serial = ctx->scene_serial;
        }
        if ((rc = ensure(ctx, d.upd_back, d.upd_back_cap, back_bytes))) return rc;
        if (back_bytes > d.h_upd_back_cap) {
            if (d.h_upd_back) cudaFreeHost(d.h_upd_back);
            d.h_upd_back = nullptr;
            d.h_upd_back_cap = 0;
            CK(ctx, cudaHostAlloc((void**)&d.h_upd_back, back_bytes, cudaHostAllocPortable));
            d.h_upd_back_cap = back_bytes;
        }
        if ((rc = ensure(ctx, d.upd_boxes, d.upd_boxes_cap, 6 * (size_t)std::max(up.n_boxed, 1)))) return rc;
        UpdateLaunch ul{};
        size_t grid_bytes = 0, tmp_bytes = 0, o_cnt = 0, o_off = 0, o_keys = 0, o_vals = 0, o_keys2 = 0, o_sorted = 0, o_items = 0, o_cc = 0,
               o_cs = 0, o_tmp = 0;
        if (grid) {
            tmp_bytes = tcrt_update_tmp_bytes(cap, n_bvh, (int)up.n_cells);
            o_cnt = carve(grid_bytes, 8 * ((size_t)n_bvh + 1));
            o_off = carve(grid_bytes, 8 * ((size_t)n_bvh + 1));
            o_keys = carve(grid_bytes, 4 * (size_t)cap);
            o_vals = carve(grid_bytes, 4 * (size_t)cap);
            o_keys2 = carve(grid_bytes, 4 * (size_t)cap);
            o_sorted = carve(grid_bytes, 4 * (size_t)cap);
            o_items = carve(grid_bytes, 4 * (size_t)cap);
            o_cc = carve(grid_bytes, 4 * (up.n_cells + 1));
            o_cs = carve(grid_bytes, 4 * (up.n_cells + 1));
            o_tmp = carve(grid_bytes, tmp_bytes);
            // the item list the scene may be reading moves only when the buffer grows (the render stream is idle here)
            if ((rc = ensure(ctx, d.upd_grid, d.upd_grid_cap, grid_bytes))) return rc;
            unsigned char* g = d.upd_grid;
            ul.grid = 1;
            for (int k = 0; k < 3; k++) {
                ul.glo[k] = up.grid.lo_d[k];
                ul.gcell[k] = up.grid.cell_d[k];
                ul.gdims[k] = up.grid.dims[k];
            }
            ul.gmargin = up.grid.reg_margin_d;
            ul.n_cells = (int)up.n_cells;
            ul.cap = cap;
            ul.reg_count = reinterpret_cast<unsigned long long*>(g + o_cnt);
            ul.reg_off = reinterpret_cast<unsigned long long*>(g + o_off);
            ul.keys = reinterpret_cast<unsigned*>(g + o_keys);
            ul.vals = reinterpret_cast<unsigned*>(g + o_vals);
            ul.keys2 = reinterpret_cast<unsigned*>(g + o_keys2);
            ul.sorted = reinterpret_cast<unsigned*>(g + o_sorted);
            ul.items = reinterpret_cast<int*>(g + o_items);
            ul.cell_count = reinterpret_cast<unsigned*>(g + o_cc);
            ul.cell_start = reinterpret_cast<unsigned*>(g + o_cs);
            ul.cells = d.scene_mem + ctx->scene_off[7];
            ul.tmp = g + o_tmp;
            ul.tmp_bytes = tmp_bytes;
            out.items[i] = ul.items;
        }
        // the input on this device (a rebox reads the blob's spheres in place: slot i is row i)
        const float4* src = rebox ? d.scene_mem : reinterpret_cast<const float4*>(geom);
        if (!rebox && (slot < 0 || d.dev != src_dev)) {
            if ((rc = ensure(ctx, d.upd_geom, d.upd_geom_cap, (size_t)n))) return rc;
            if (slot < 0)
                CK(ctx, cudaMemcpyAsync(d.upd_geom, ctx->upd_stage, (size_t)n * sizeof(float4), cudaMemcpyHostToDevice, d.stream));
            else
                CK(ctx, cudaMemcpyPeerAsync(d.upd_geom, d.dev, geom, src_dev, (size_t)n * sizeof(float4), d.stream));
            src = d.upd_geom;
        }
        ul.geom = src;
        ul.n = n;
        ul.slot_of = rebox ? d.upd_maps + o_ident : d.upd_maps;
        ul.spheres = d.scene_mem;
        ul.n_boxed = up.n_boxed;
        ul.n_bvh = n_bvh;
        ul.ext_fixed = ext_fixed;
        ul.light_sph = rebox ? d.upd_maps + o_ident + n : d.upd_maps + n;
        ul.n_light_sph = n_ls;
        ul.back = reinterpret_cast<UpdateBack*>(d.upd_back);
        ul.boxes = d.upd_boxes;
        if (ctx->scene_bvh_s) {
            ul.nodes = d.scene_mem + ctx->scene_off[5];
            ul.levels = d.upd_maps + n + n_ls;
            ul.level_start = ul.levels + up.levels.size();
            ul.n_levels = n_levels;
        }
        CK(ctx, cudaEventRecord(d.ev_u0, d.stream));
        CK(ctx, tcrt_launch_update_spheres(ul, d.sm_count, d.stream, launches));
        CK(ctx, cudaEventRecord(d.ev_u1, d.stream));
        CK(ctx, cudaMemcpyAsync(d.h_upd_back, d.upd_back, back_bytes, cudaMemcpyDeviceToHost, d.stream));
    }
    bool invalid = false;
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));
        CK(ctx, cudaEventElapsedTime(&out.ms[i], d.ev_u0, d.ev_u1));
        invalid = invalid || reinterpret_cast<const UpdateBack*>(d.h_upd_back)->invalid != 0;
    }
    out.invalid = invalid;
    if (invalid && rebox) return TCRT_OK;   // the upload does not check spheres; their boxes stay as they are
    if (invalid)   // no launch after the check wrote anything: the scene is unchanged
        return fail(ctx, TCRT_ERR_INVALID, "sphere_geom holds a centre or radius_squared that is not finite, or radius_squared < 0");

    // the bounds and the light positions (every device reduced the same values)
    const UpdateBack& b = *reinterpret_cast<const UpdateBack*>(ctx->devs[0].h_upd_back);
    auto unkey = [](unsigned key) {
        const unsigned u = (key & 0x80000000u) ? (key & 0x7fffffffu) : ~key;
        float f;
        memcpy(&f, &u, 4);
        return f;
    };
    SceneBounds& bounds = out.bounds;
    bounds = up.bounds;
    for (int k = 0; k < 3; k++) {
        if (b.lo_key[k]) bounds.sph_lo[k] = unkey(~b.lo_key[k]);
        if (b.hi_key[k]) bounds.sph_hi[k] = unkey(b.hi_key[k]);
    }
    if (n_bvh > 0) {
        const unsigned r2 = ~b.r2min_key;
        float r2f;
        memcpy(&r2f, &r2, 4);
        bounds.rmin = sqrtf(r2f);
    }
    float ext_sph;
    memcpy(&ext_sph, &b.ext_bits, 4);
    out.ext_sph = ext_sph;
    out.keep_grid = grid && !b.grid_out && !b.grid_full;
    const float* centres = reinterpret_cast<const float*>(&b + 1);
    out.og = up.light_og;
    for (int j = 0; j < n_ls; j++)
        for (int k = 0; k < 3; k++) out.og[3 * up.light_of_sph[j] + k] = centres[3 * j + k];
    return TCRT_OK;
}

// The per-launch scalars of ds into every device's scene, and the grid as the sphere launches left it
static void set_scalars(tcrt_ctx* ctx, const DeviceScene& ds, bool keep_grid, const std::vector<int*>& items) {
    for (size_t i = 0; i < ctx->devs.size(); i++) {
        DeviceScene& dd = ctx->devs[i].ds;
        dd.bvh_cx = ds.bvh_cx; dd.bvh_cy = ds.bvh_cy; dd.bvh_cz = ds.bvh_cz;
        dd.bvh_r2 = ds.bvh_r2; dd.bvh_rmin = ds.bvh_rmin; dd.bvh_cmax = ds.bvh_cmax;
        dd.clu_cx = ds.clu_cx; dd.clu_cy = ds.clu_cy; dd.clu_cz = ds.clu_cz; dd.clu_rbig = ds.clu_rbig;
        dd.grid_k2_max = ds.grid_k2_max;
        if (!items.empty()) dd.grid_items = keep_grid ? items[i] : nullptr;
        if (!keep_grid) dd.grid_cells = nullptr;
    }
}

static int update_impl(tcrt_ctx* ctx, int slot, const float* geom, tcrt_stats* stats) {
    if (!ctx || !geom) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    const int nd = (int)ctx->devs.size();
    if (slot >= 0) {
        if (slot >= nd) return fail(ctx, TCRT_ERR_INVALID, "device slot %d out of range (have %d)", slot, nd);
        const int src_dev = ctx->devs[slot].dev;
        if (!on_device(geom, src_dev)) return fail(ctx, TCRT_ERR_INVALID, "sphere_geom is not device memory of slot %d's device", slot);
        if (reinterpret_cast<uintptr_t>(geom) % 16 != 0)   // the launches read it as float4
            return fail(ctx, TCRT_ERR_INVALID, "sphere_geom is not 16-byte aligned");
    }
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        stats->n_devices = nd;
    }
    UpdatePlan& up = ctx->scene_upd;
    if (up.n_spheres == 0) return TCRT_OK;
    int launches = 0;
    SpherePass sp;
    if (int rc = sphere_pass(ctx, slot, geom, false, up.ext_fixed, sp, &launches)) return rc;

    // the scalars and the light rows, with the upload's code
    DeviceScene ds = ctx->scene_ds;
    scene_scalars(sp.bounds, ctx->scene_bvh_s, !up.clusters.empty(), sp.keep_grid, ds);
    for (int l = 0; l < ds.n_lights; l++)
        light_rows(&sp.og[3 * l], up.light_int[l], &up.light_col[3 * l], up.clusters, ds, ctx->upd_stage + 2 * l);
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        CK(ctx, cudaSetDevice(d.dev));
        if (ds.n_lights > 0)
            CK(ctx, cudaMemcpyAsync(d.scene_mem + ds.light_off, ctx->upd_stage, 2 * (size_t)ds.n_lights * sizeof(float4),
                                    cudaMemcpyHostToDevice, d.stream));
    }
    set_scalars(ctx, ds, sp.keep_grid, sp.items);
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));
        if (stats) stats->render_ms[i] = sp.ms[i];
    }
    if (stats) stats->gpu_launches = (unsigned long long)launches;
    // what a later plane update starts from
    up.bounds = sp.bounds;
    up.light_og = sp.og;
    up.ext_sph = sp.ext_sph;
    up.ext_sph_box = scene_ext(up.ext_fixed, sp.ext_sph);
    ctx->scene_ds = ds;
    ctx->scene_grid = sp.keep_grid;
    ctx->scene_key.clear();        // the staged blob no longer matches the devices: the next upload rebuilds
    ctx->cut_valid = false;
    ctx->costs_valid = false;
    return TCRT_OK;
}

extern "C" {

int tcrt_update_spheres(tcrt_ctx* ctx, const float* sphere_geom, tcrt_stats* stats) {
    return update_impl(ctx, -1, sphere_geom, stats);
}

int tcrt_update_spheres_device(tcrt_ctx* ctx, int device_slot, const float* sphere_geom, tcrt_stats* stats) {
    if (ctx && device_slot < 0) return fail(ctx, TCRT_ERR_INVALID, "device slot %d out of range", device_slot);
    return update_impl(ctx, device_slot, sphere_geom, stats);
}

}  // extern "C"

// ---- material edits (tcrt_update_materials, tcrt_update_textures) ------------------------------------------------------------
// New colours, shading factors, intensities, texture ids and checker rows for the resident scene.  The host checks the input
// against its copy of the materials (ctx->scene_mat) before anything changes, merges it in and packs full rows;
// tcrt_materials.cu scatters them on every device.  The dead-path bound is the only host state derived from materials, and
// it is recomputed from the copy.  DESIGN.md §4.3.

// The n records packed in ctx->upd_stage -> every device: one copy and one scatter launch each, on the render stream after
// the frames queued before the call.
static int send_material_records(tcrt_ctx* ctx, int n, tcrt_stats* stats) {
    const MaterialShadow& m = ctx->scene_mat;
    const int nd = (int)ctx->devs.size();
    int launches = 0;
    for (auto& d : ctx->devs) {
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));   // frames queued before the call finish with the old materials
        if (!d.ev_u0) CK(ctx, cudaEventCreate(&d.ev_u0));
        if (!d.ev_u1) CK(ctx, cudaEventCreate(&d.ev_u1));
        int rc = ensure(ctx, d.mat_light_of, d.mat_light_of_cap, std::max(m.light_of.size(), (size_t)1));
        if (rc) return rc;
        if (d.mat_serial != ctx->scene_serial) {   // the map, once per upload
            CK(ctx, cudaMemcpy(d.mat_light_of, m.light_of.data(), m.light_of.size() * sizeof(int), cudaMemcpyHostToDevice));
            d.mat_serial = ctx->scene_serial;
        }
        if ((rc = ensure(ctx, d.mat_rec, d.mat_rec_cap, (size_t)n))) return rc;
        CK(ctx, cudaMemcpyAsync(d.mat_rec, ctx->upd_stage, (size_t)n * sizeof(MaterialRecord), cudaMemcpyHostToDevice, d.stream));
        MaterialLaunch ml{};
        ml.rec = d.mat_rec;
        ml.n = n;
        ml.surface = d.scene_mem + ctx->scene_off[0];
        ml.material = d.scene_mem + ctx->scene_off[1];
        ml.textures = d.scene_mem + ctx->scene_off[4];
        ml.lights = d.scene_mem + ctx->scene_ds.light_off;
        ml.light_of = d.mat_light_of;
        CK(ctx, cudaEventRecord(d.ev_u0, d.stream));
        CK(ctx, tcrt_launch_material_edit(ml, d.stream, &launches));
        CK(ctx, cudaEventRecord(d.ev_u1, d.stream));
    }
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));
        if (stats) {
            float ms = 0.f;
            CK(ctx, cudaEventElapsedTime(&ms, d.ev_u0, d.ev_u1));
            stats->render_ms[i] = ms;
        }
    }
    if (stats) stats->gpu_launches = (unsigned long long)launches;
    const tcrt_scene view = m.view();
    ctx->scene_dead = dead_path_bound(&view);
    ctx->scene_key.clear();        // the staged blob no longer matches the devices: the next upload rebuilds
    ctx->cut_valid = false;        // bounce counts follow the reflective factors and the dead paths
    ctx->costs_valid = false;
    return TCRT_OK;
}

static void clear_stats(tcrt_ctx* ctx, tcrt_stats* stats) {
    if (!stats) return;
    memset(stats, 0, sizeof(*stats));
    stats->n_devices = (int)ctx->devs.size();
}

extern "C" {

int tcrt_update_materials(tcrt_ctx* ctx, int n, const int* objects, const float* surface, const float* material,
                          const int* texture, tcrt_stats* stats) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (n < 0) return fail(ctx, TCRT_ERR_INVALID, "n = %d is negative", n);
    if (!surface && !material && !texture) return fail(ctx, TCRT_ERR_INVALID, "surface, material and texture are all NULL");
    if (n > 0 && !objects) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    MaterialShadow& m = ctx->scene_mat;
    const int n_obj = m.n_objects(), n_tex = m.n_textures();
    std::vector<char> seen(n_obj, 0);
    for (int i = 0; i < n; i++) {
        const int o = objects[i];
        if (o < 0 || o >= n_obj) return fail(ctx, TCRT_ERR_INVALID, "object index %d out of range (have %d)", o, n_obj);
        if (seen[o]) return fail(ctx, TCRT_ERR_INVALID, "object %d is listed twice", o);
        seen[o] = 1;
        if (texture && (texture[i] < -1 || texture[i] >= n_tex))
            return fail(ctx, TCRT_ERR_INVALID, "texture id %d out of range (have %d)", texture[i], n_tex);
    }
    clear_stats(ctx, stats);
    if (n == 0) return TCRT_OK;
    if (int rc = ensure_upd_stage(ctx, sizeof(MaterialRecord) / sizeof(float4) * (size_t)n)) return rc;
    MaterialRecord* rec = reinterpret_cast<MaterialRecord*>(ctx->upd_stage);
    UpdatePlan& up = ctx->scene_upd;
    for (int i = 0; i < n; i++) {
        const int o = objects[i];
        float* sf = &m.surface[4 * (size_t)o];
        float* mt = &m.material[4 * (size_t)o];
        if (surface) memcpy(sf, surface + 4 * (size_t)i, 4 * sizeof(float));
        if (material) memcpy(mt, material + 4 * (size_t)i, 3 * sizeof(float));   // w is not a material
        if (texture) m.info[4 * (size_t)o + 3] = texture[i];
        rec[i] = MaterialRecord{};
        rec[i].a = make_float4(sf[0], sf[1], sf[2], sf[3]);
        rec[i].b = make_float4(mt[0], mt[1], mt[2], mt[3]);
        rec[i].target = o;
        rec[i].tex = m.info[4 * (size_t)o + 3];
        const int l = m.light_of[o];
        if (l >= 0) {   // tcrt_update_spheres rewrites every light row from these
            for (int k = 0; k < 3; k++) up.light_col[3 * l + k] = sf[k];
            up.light_int[l] = mt[2];
        }
    }
    return send_material_records(ctx, n, stats);
}

int tcrt_update_textures(tcrt_ctx* ctx, int n, const int* textures, const float* rows, tcrt_stats* stats) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (n < 0) return fail(ctx, TCRT_ERR_INVALID, "n = %d is negative", n);
    if (n > 0 && (!textures || !rows)) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    MaterialShadow& m = ctx->scene_mat;
    const int n_tex = m.n_textures();
    std::vector<char> seen(n_tex, 0);
    for (int i = 0; i < n; i++) {
        const int t = textures[i];
        if (t < 0 || t >= n_tex) return fail(ctx, TCRT_ERR_INVALID, "texture id %d out of range (have %d)", t, n_tex);
        if (seen[t]) return fail(ctx, TCRT_ERR_INVALID, "texture %d is listed twice", t);
        seen[t] = 1;
    }
    clear_stats(ctx, stats);
    if (n == 0) return TCRT_OK;
    if (int rc = ensure_upd_stage(ctx, sizeof(MaterialRecord) / sizeof(float4) * (size_t)n)) return rc;
    MaterialRecord* rec = reinterpret_cast<MaterialRecord*>(ctx->upd_stage);
    for (int i = 0; i < n; i++) {
        const int t = textures[i];
        const float* row = rows + 8 * (size_t)i;
        memcpy(&m.textures[8 * (size_t)t], row, 8 * sizeof(float));
        rec[i] = MaterialRecord{};
        rec[i].a = make_float4(row[0], row[1], row[2], row[3]);
        rec[i].b = make_float4(row[4], row[5], row[6], row[7]);
        rec[i].target = ~t;
        rec[i].tex = -1;
    }
    return send_material_records(ctx, n, stats);
}

}  // extern "C"

// ---- moving planes (tcrt_update_planes) --------------------------------------------------------------------------------------
// New rows for finite and infinite planes of the resident scene.  Planes are few (every finite plane is staged in shared
// memory), so the host plans from its copy of the finite-plane rows (UpdatePlan) with the upload's own code: plane and
// normal rows, the finite-plane BVH's leaf boxes (fin_box), the clusters' hulls (tcrt_refit_box_cluster) or their drop,
// the light table (light_rows) and the per-launch scalars (scene_scalars).  tcrt_update.cu scatters the rows and refits
// the finite-plane BVH.  When the new plane origins raise ext above the ext the resident sphere boxes were built with, the
// sphere update's launches box the resident spheres again first.  DESIGN.md §4.3, §4.5.

extern "C" int tcrt_update_planes(tcrt_ctx* ctx, int n, const int* objects, const float* geom, const float* normals,
                                  const float* origin, tcrt_stats* stats) {
    if (!ctx) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (n < 0) return fail(ctx, TCRT_ERR_INVALID, "n = %d is negative", n);
    if (n > 0 && (!objects || !geom || !normals || !origin)) return fail(ctx, TCRT_ERR_INVALID, "null argument");
    if (!ctx->has_scene) return fail(ctx, TCRT_ERR_NO_SCENE, "tcrt_upload_scene has not been called");
    UpdatePlan& up = ctx->scene_upd;
    const int n_obj = ctx->n_objects;
    std::vector<char> seen(n_obj, 0);
    for (int i = 0; i < n; i++) {
        const int o = objects[i];
        if (o < 0 || o >= n_obj) return fail(ctx, TCRT_ERR_INVALID, "object index %d out of range (have %d)", o, n_obj);
        if (up.fin_slot_of_obj[o] < 0 && up.inf_slot_of_obj[o] < 0)
            return fail(ctx, TCRT_ERR_INVALID, "object %d is a sphere (tcrt_update_spheres moves spheres)", o);
        if (seen[o]) return fail(ctx, TCRT_ERR_INVALID, "object %d is listed twice", o);
        seen[o] = 1;
    }
    clear_stats(ctx, stats);
    if (n == 0) return TCRT_OK;
    const int nd = (int)ctx->devs.size();
    const MaterialShadow& mat = ctx->scene_mat;
    DeviceScene ds = ctx->scene_ds;

    // the rows of the moved planes, into the host's copy and the records
    std::vector<PlaneRecord> rec;
    auto put = [&](size_t dst, float4 v) {
        PlaneRecord r{};
        r.v = v;
        r.dst = (int)dst;
        rec.push_back(r);
    };
    auto f4 = [](const float* p) { return make_float4(p[0], p[1], p[2], p[3]); };
    std::vector<int> moved_fin;   // finite-plane slots of the moved non-light planes
    for (int i = 0; i < n; i++) {
        const int o = objects[i];
        const float* g = geom + 16 * (size_t)i;
        const int fs = up.fin_slot_of_obj[o], is = up.inf_slot_of_obj[o];
        if (fs >= 0) {
            memcpy(&up.fin_rows[16 * (size_t)fs], g, 16 * sizeof(float));
            for (int j = 0; j < 4; j++) put((size_t)ds.fin_off + 4 * (size_t)fs + j, f4(g + 4 * j));
            if (fs < ds.n_fin_nl) moved_fin.push_back(fs);
        } else {
            put((size_t)ds.inf_off + is, f4(g));
            for (int j = 0; j < 3; j++) put(up.off_frame + 3 * (size_t)is + j, f4(g + 4 * (j + 1)));
        }
        float4 nr[6];
        normal_rows(normals + 8 * (size_t)i, nr);
        for (int k = 0; k < 6; k++) put(up.off_normals + 6 * (size_t)o + k, nr[k]);
        const int l = mat.light_of[o];
        if (l >= 0)
            for (int k = 0; k < 3; k++) up.light_og[3 * (size_t)l + k] = origin[4 * (size_t)i + k];
    }

    // ext of the moved scene: its finite-plane origins and the spheres' extent of the last read-back
    double ext_fixed = 1.0;
    for (int k = 0; k < ds.n_fin; k++)
        for (int c = 0; c < 3; c++) ext_fixed = std::max(ext_fixed, fabs((double)up.fin_rows[16 * (size_t)k + 12 + c]));
    const double ext = scene_ext(ext_fixed, up.ext_sph);

    // the planes' part of the bounds: the finite-plane BVH's leaf boxes and the clusters' hulls
    SceneBounds bounds = up.bounds;
    for (int k = 0; k < 3; k++) {
        bounds.pl_lo[k] = 1e300;
        bounds.pl_hi[k] = -1e300;
    }
    const int nb = ctx->scene_bvh_f ? ds.n_fin_bvh : 0;
    if (nb > 0) {
        // every resident box at least as wide as the upload of the moved scene makes it: all of them again when ext grew
        const double margin = 1e-5 * ext;
        if (ext > up.ext_fin_box) {
            for (int k = 0; k < nb; k++) fin_box(&up.fin_rows[16 * (size_t)k], margin, &up.fin_boxes[6 * (size_t)k]);
            up.ext_fin_box = ext;
        } else {
            for (int k : moved_fin)
                if (k < nb) fin_box(&up.fin_rows[16 * (size_t)k], margin, &up.fin_boxes[6 * (size_t)k]);
            up.ext_fin_box = std::min(up.ext_fin_box, ext);
        }
        for (int k = 0; k < nb; k++) grow_into(bounds.pl_lo, bounds.pl_hi, &up.fin_boxes[6 * (size_t)k]);
    }
    std::vector<TcrtBoxCluster> clusters = up.clusters;
    for (TcrtBoxCluster& c : clusters)
        if (!tcrt_refit_box_cluster(up.fin_rows.data(), c)) {
            // a member left its face's axis: no cluster until the next upload.  The rectangles already sit after the
            // generic planes, so the linear sweep over [0, n_fin_nl) takes them (FM 3).
            clusters.clear();
            ds.n_clu = 0;
            ds.n_arect = 0;
            ds.n_fin_gen = ds.n_fin_nl;
            break;
        }
    for (int c = 0; c < (int)clusters.size(); c++) {
        grow_into(bounds.pl_lo, bounds.pl_hi, clusters[c].lo);   // lo[3], hi[3] are contiguous: a 6-float box
        float4 rows[4];
        cluster_rows(clusters[c], rows);
        for (int j = 0; j < 4; j++) put((size_t)ds.clu_off + 4 * (size_t)c + j, rows[j]);
    }

    // the spheres boxed again when ext grew past the ext of their boxes (a lower ext keeps the wider boxes, still sound)
    int launches = 0;
    SpherePass sp;
    bool rebox = up.n_boxed > 0 && ext > up.ext_sph_box;
    if (rebox) {
        if (int rc = sphere_pass(ctx, -1, nullptr, true, ext_fixed, sp, &launches)) return rc;
        rebox = !sp.invalid;
    }
    if (rebox) {
        for (int k = 0; k < 3; k++) {
            bounds.sph_lo[k] = sp.bounds.sph_lo[k];
            bounds.sph_hi[k] = sp.bounds.sph_hi[k];
        }
        bounds.rmin = sp.bounds.rmin;
    }
    const bool keep_grid = rebox ? sp.keep_grid : ctx->scene_grid;

    // the scalars and every light row, with the upload's code
    scene_scalars(bounds, ctx->scene_bvh_s, !clusters.empty(), keep_grid, ds);
    for (int l = 0; l < ds.n_lights; l++) {
        float4 rows[2];
        light_rows(&up.light_og[3 * (size_t)l], up.light_int[l], &up.light_col[3 * (size_t)l], clusters, ds, rows);
        put((size_t)ds.light_off + 2 * (size_t)l, rows[0]);
        put((size_t)ds.light_off + 2 * (size_t)l + 1, rows[1]);
    }

    // every device: the records (and the leaf boxes), one scatter launch, the refit
    const size_t rec_f4 = rec.size() * (sizeof(PlaneRecord) / sizeof(float4));
    const int n_levels = nb > 0 ? (int)up.fin_level_start.size() - 1 : 0;
    if (int rc = ensure_upd_stage(ctx, rec_f4 + (6 * (size_t)nb + 3) / 4)) return rc;
    memcpy(ctx->upd_stage, rec.data(), rec.size() * sizeof(PlaneRecord));
    float* boxes_stage = reinterpret_cast<float*>(ctx->upd_stage + rec_f4);
    if (nb > 0) memcpy(boxes_stage, up.fin_boxes.data(), 6 * (size_t)nb * sizeof(float));
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));   // frames queued before the call finish with the old planes
        if (!d.ev_u0) CK(ctx, cudaEventCreate(&d.ev_u0));
        if (!d.ev_u1) CK(ctx, cudaEventCreate(&d.ev_u1));
        int rc = ensure(ctx, d.pl_rec, d.pl_rec_cap, rec.size());
        if (rc) return rc;
        CK(ctx, cudaMemcpyAsync(d.pl_rec, ctx->upd_stage, rec.size() * sizeof(PlaneRecord), cudaMemcpyHostToDevice, d.stream));
        PlaneLaunch pl{};
        pl.rec = d.pl_rec;
        pl.n = (int)rec.size();
        pl.scene = d.scene_mem;
        if (n_levels > 0) {
            const size_t n_lv = up.fin_levels.size() + up.fin_level_start.size();
            if ((rc = ensure(ctx, d.pl_levels, d.pl_levels_cap, n_lv))) return rc;
            if (d.pl_serial != ctx->scene_serial) {   // the levels, once per upload
                std::vector<int> lv(up.fin_levels);
                lv.insert(lv.end(), up.fin_level_start.begin(), up.fin_level_start.end());
                CK(ctx, cudaMemcpy(d.pl_levels, lv.data(), lv.size() * sizeof(int), cudaMemcpyHostToDevice));
                d.pl_serial = ctx->scene_serial;
            }
            if ((rc = ensure(ctx, d.pl_boxes, d.pl_boxes_cap, 6 * (size_t)nb))) return rc;
            if ((rc = ensure(ctx, d.upd_back, d.upd_back_cap, sizeof(UpdateBack)))) return rc;
            CK(ctx, cudaMemcpyAsync(d.pl_boxes, boxes_stage, 6 * (size_t)nb * sizeof(float), cudaMemcpyHostToDevice, d.stream));
            pl.boxes = d.pl_boxes;
            pl.nodes = d.scene_mem + ctx->scene_off[6];
            pl.levels = d.pl_levels;
            pl.level_start = d.pl_levels + up.fin_levels.size();
            pl.n_levels = n_levels;
            pl.back = reinterpret_cast<UpdateBack*>(d.upd_back);
        }
        CK(ctx, cudaEventRecord(d.ev_u0, d.stream));
        CK(ctx, tcrt_launch_update_planes(pl, d.stream, &launches));
        CK(ctx, cudaEventRecord(d.ev_u1, d.stream));
    }
    set_scalars(ctx, ds, keep_grid, rebox ? sp.items : std::vector<int*>());
    for (int i = 0; i < nd; i++) {
        DeviceState& d = ctx->devs[i];
        d.ds.n_clu = ds.n_clu;
        d.ds.n_arect = ds.n_arect;
        d.ds.n_fin_gen = ds.n_fin_gen;
        CK(ctx, cudaSetDevice(d.dev));
        CK(ctx, cudaStreamSynchronize(d.stream));
        if (stats) {
            float ms = 0.f;
            CK(ctx, cudaEventElapsedTime(&ms, d.ev_u0, d.ev_u1));
            stats->render_ms[i] = ms + (rebox ? sp.ms[i] : 0.f);
        }
    }
    if (stats) stats->gpu_launches = (unsigned long long)launches;
    // what later updates start from
    up.ext_fixed = ext_fixed;
    if (rebox) up.ext_sph_box = ext;
    up.bounds = bounds;
    up.clusters.swap(clusters);
    ctx->scene_ds = ds;
    ctx->scene_grid = keep_grid;
    ctx->scene_key.clear();        // the staged blob no longer matches the devices: the next upload rebuilds
    ctx->cut_valid = false;
    ctx->costs_valid = false;
    return TCRT_OK;
}
