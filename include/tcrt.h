/* include/tcrt.h — C ABI of the B200 render path (libtcrt.so).
 *
 * The reference (ccelio/TileCodeRayTracer) has no plugin / FFI boundary: it is one
 * executable whose hot path is
 *     the pixel double loop                RayTracer.cpp:911-923   (createEyeRay + calculatePixel)
 *     calculatePixel / getCollision /      RayTracer.cpp:448-638, :50-89,
 *       cosineShade / inShade                :654-701, :709-771
 *     SceneObject::collision (3 types)     SceneSphere.cpp:50-168, SceneInfinitePlane.cpp:29-108,
 *                                          SceneFinitePlane.cpp:86-164
 *     the .txt writer                      RayTracer.cpp:2022-2061 (init_log), :1574-1626 (printPixelsToLog)
 * This header is the boundary a maintainer would bind instead of those call sites
 * (INTEGRATION.md shows the binding).  Plain pointers and sizes only; the caller owns
 * every input array and every output buffer, the library owns device memory inside
 * tcrt_ctx.  Errors are returned as negative ints (the reference returns 0 ok / 1 error
 * from init_log / raytrace_main, RayTracer.cpp:862-873,2027-2031) and never cross the
 * boundary as exceptions or exit().  One ctx is used from one host thread at a time.
 *
 * There is no CPU fallback anywhere behind this API: with no usable CUDA device every
 * entry point that needs one fails with TCRT_ERR_NO_DEVICE.
 */
#ifndef TCRT_H_
#define TCRT_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TCRT_ABI_VERSION 2
#define TCRT_MAX_DEVICES 16

enum {
    TCRT_OK = 0,
    TCRT_ERR_INVALID = -1,     /* bad argument */
    TCRT_ERR_CUDA = -2,        /* a CUDA runtime call failed; see tcrt_last_error */
    TCRT_ERR_NO_DEVICE = -3,   /* no CUDA device / device id out of range */
    TCRT_ERR_IO = -4,          /* fopen / write failed */
    TCRT_ERR_NO_SCENE = -5,    /* render before tcrt_upload_scene */
    TCRT_ERR_NO_FRAME = -6,    /* download / format before a render */
    TCRT_ERR_UNSUPPORTED = -7  /* e.g. max_depth above TCRT_MAX_DEPTH */
};

/* Deepest recursion cap the kernels are instantiated for (reference ships 50,
 * rt_project_parameters.h:73). */
#define TCRT_MAX_DEPTH 254

typedef struct tcrt_ctx tcrt_ctx; /* opaque */

/* Object types, in the order the kernels sweep them. */
enum { TCRT_SPHERE = 0, TCRT_FINITE_PLANE = 1, TCRT_INFINITE_PLANE = 2 };

/* ---- flattened scene ------------------------------------------------------------
 * What Scene::flatten() (include/CelioRayTracer.hpp) exports: the reference's
 * SceneObject* list (Scene.h:36, virtual collision() per object) turned into per-type
 * structure-of-arrays.  All floats are IEEE binary32 exactly as the reference's ctors
 * leave them in the objects' private members (normalised normals, r*r, -(o.n), ...);
 * nothing is re-derived on the device.  "object index" = position in the Scene's list;
 * it decides nearest-hit ties (first strictly-smaller distance wins, RayTracer.cpp:73-86)
 * and the light loop order (RayTracer.cpp:540-544).
 * Within each type, primitives appear in increasing object index.                      */
typedef struct tcrt_scene {
    int n_objects;
    int n_spheres;
    int n_fin_planes;
    int n_inf_planes;
    int n_lights;
    int n_textures;

    /* SceneSphere (SceneSphere.h:17-19): centre xyz, radius_squared.        [n_spheres][4] */
    const float* sphere_geom;
    const int* sphere_obj; /* object index                                   [n_spheres]    */

    /* SceneFinitePlane (SceneFinitePlane.h:32-45), 4 x float4 per plane:
     *   (normal xyz, -distance_to_origin) (horizontal xyz, h_distance)
     *   (vertical xyz, v_distance)        (plane_origin xyz, 0)             [n_fin_planes][16] */
    const float* fin_geom;
    const int* fin_obj; /*                                                   [n_fin_planes]  */

    /* SceneInfinitePlane (SceneInfinitePlane.h:24-31), 4 x float4 per plane:
     *   (normal xyz, -distance_to_origin) (horizontal xyz, 0)
     *   (vertical xyz, 0)                 (SceneObject origin xyz, 0)       [n_inf_planes][16] */
    const float* inf_geom;
    const int* inf_obj; /*                                                   [n_inf_planes]  */

    /* Per object, indexed by object index (winner-only data):
     *   obj_surface  (colour r g b, diffuse_factor)      ObjMaterial.h:70-80    [n_objects][4]
     *   obj_material (specular, reflective, intensity, 0) SceneObject.h:191-194 [n_objects][4]
     *   obj_origin   (SceneObject::origin xyz, 0) — the light position         [n_objects][4]
     *   obj_normals  (facing normal xyz,0, reverseNormal xyz,0); zeros for spheres.  For
     *                finite planes reverseNormal is -normal re-normalised
     *                (SceneFinitePlane.cpp:34-35,65-66), for infinite planes plain -normal
     *                (SceneInfinitePlane.cpp:23).                              [n_objects][8]
     *   obj_info     (type, slot within its type array, is_light, texture id or -1) [n_objects][4] */
    const float* obj_surface;
    const float* obj_material;
    const float* obj_origin;
    const float* obj_normals;
    const int* obj_info;

    const int* light_obj; /* object indices of lights, increasing            [n_lights] */

    /* Texture_CheckerBoard (Texture_CheckerBoard.h:23-71):
     *   (light r g b, width) (dark r g b, height)                           [n_textures][8] */
    const float* textures;
} tcrt_scene;

/* Camera (Camera.h:20-39, Camera.cpp:9-40): everything createEyeRay (Camera.cpp:71-84) reads. */
typedef struct tcrt_camera {
    float eye[3];           /* eye_origin */
    float screen_origin[3];
    float horizontal[3];    /* vector_horizontal, normalised */
    float vertical[3];      /* vector_vertical, normalised */
    float screen_width, screen_height;
    float screen_halfwidth, screen_halfheight;
} tcrt_camera;

/* The reference's compile-time knobs (rt_project_parameters.h:24-25,65-66,73-74;
 * NULL_COLOR RayTracer.h:52) as run-time parameters. */
typedef struct tcrt_params {
    int width;          /* SCREEN_HORIZONTAL_RESOLUTION */
    int height;         /* SCREEN_VERTICAL_RESOLUTION */
    int max_depth;      /* MAX_RECURSION_LEVEL: levels 0..max_depth are traced */
    int shadows_on;     /* SHADOWS_ON */
    int reflections_on; /* REFLECTIONS_ON */
    float null_color[3];/* NULL_COLOR (0.75,0.75,0.75): miss / recursion cap */
    float far_dist;     /* FLOAT_MAX_VALUE 65535: hits at or beyond are invisible.  Any value is
                         * accepted and rendered like the reference: +inf sees every hit; at
                         * far_dist <= 0 only a sphere around the ray's origin (its distance is
                         * negative) can still be hit; -inf and NaN hide everything. */
} tcrt_params;

/* Fills the reference's shipped values: 500x504, depth 50, shadows+reflections on,
 * grey 0.75, far 65535. */
void tcrt_default_params(tcrt_params* p);

typedef struct tcrt_stats {
    int n_devices;
    int col_begin[TCRT_MAX_DEVICES]; /* band [col_begin, col_end) rendered by each device */
    int col_end[TCRT_MAX_DEVICES];
    double render_ms[TCRT_MAX_DEVICES]; /* kernel time, CUDA events on the launching stream (RGB8 frames: render +
                                           quantisation; supersampled frames: render + resolve) */
    double d2h_ms[TCRT_MAX_DEVICES];    /* copy-back time of the band (0 if none) */
    unsigned long long rays_primary[TCRT_MAX_DEVICES];
    unsigned long long rays_shadow[TCRT_MAX_DEVICES];
    unsigned long long rays_reflect[TCRT_MAX_DEVICES];
    unsigned long long gpu_launches;    /* kernels launched by this call (RGB8 frames: the quantisation launches too;
                                           supersampled frames: the resolve launches too) */
} tcrt_stats;

/* ---- context ------------------------------------------------------------------- */
int tcrt_abi_version(void);
int tcrt_device_count(void); /* >=0, or TCRT_ERR_NO_DEVICE */
/* device_ids == NULL: devices 0..n_devices-1.  A multi-device ctx splits every render
 * into one band of columns per device (SURVEY §8e; reference strategy 1,
 * RayTracer.cpp:904-906, with the band axis turned so a band is contiguous in the
 * x-major pixel array). */
int tcrt_create(tcrt_ctx** out, const int* device_ids, int n_devices);
void tcrt_destroy(tcrt_ctx* ctx);
const char* tcrt_last_error(tcrt_ctx* ctx); /* never NULL; ctx may be NULL */

/* Pinned host memory for output buffers (optional; pageable buffers work, slower). */
void* tcrt_alloc_host(size_t bytes);
void tcrt_free_host(void* p);

/* ---- scene ---------------------------------------------------------------------- */
/* Copies scene + camera to every device of the ctx.  Replaces: Scene::initialize() being
 * visible to calculatePixel through the global my_scene / my_camera (RayTracer.h:50-51). */
int tcrt_upload_scene(tcrt_ctx* ctx, const tcrt_scene* scene, const tcrt_camera* camera);

/* Which pruning structures the uploaded scene got (none of them can change a result; tests assert that the intended
 * kernel path is exercised): info[0] spheres in the sphere BVH, [1] cells of the uniform sphere grid (0: none), [2] finite
 * planes in their BVH, [3] box clusters, [4] rectangles owned by clusters, [5] spheres swept linearly, [6] finite planes
 * swept linearly, [7] bytes of scene staged into shared memory per CTA. */
int tcrt_scene_structures(tcrt_ctx* ctx, int info[8]);
/* The same decision for a scene that has not been uploaded — host work only, no device needed (sort, box clusters, BVHs,
 * grid; what tcrt_upload_scene does before its copy).  grid_dims (optional): cells per axis of the sphere grid, 0 0 0
 * without one.  TCRT_ERR_UNSUPPORTED for a scene tcrt_upload_scene would refuse. */
int tcrt_plan_scene(const tcrt_scene* scene, int info[8], int grid_dims[3]);
/* Host only, for tests of the grid's soundness (DESIGN.md 4.5): for each of n_points points (x, y, z), the object
 * indices of the spheres registered in the cell of the sphere grid that contains it — objects[i*cap .. i*cap + cap),
 * counts[i] of them (0 outside the grid's box).  TCRT_ERR_UNSUPPORTED when the scene gets no grid.  grid_margin
 * (optional): the fattening up to which a ray may use the grid. */
int tcrt_plan_grid_cells(const tcrt_scene* scene, const float* points, int n_points, int* objects, int cap, int* counts,
                         float* grid_margin);
/* Host only: *prune = 1 when renders of the scene with params may skip the shading of reflection levels whose colour the
 * reference multiplies by zero (the path's every channel has met a zero object colour above them; sphere-grid scenes,
 * DESIGN.md 4.1c) — when a bound on every colour the reference forms on the way is finite and far from overflow.  The
 * result is the same either way; 0 where a zero could meet an overflowed colour and make NaN, which is then rendered.
 * Bad params: TCRT_ERR_INVALID; max_depth above TCRT_MAX_DEPTH: TCRT_ERR_UNSUPPORTED, as for renders. */
int tcrt_plan_dead_paths(const tcrt_scene* scene, const tcrt_params* params, int* prune);

/* ---- render (replaces the pixel loop RayTracer.cpp:911-923) ----------------------- */
/* Whole image -> host_rgb[width*height*3], x-major, z fastest, (r,g,b) float32: the layout
 * of the reference's pixels[W][H] (RayTracer.h:44).  stats may be NULL.  host_rgb may be pinned (tcrt_alloc_host,
 * cudaHostAlloc: column chunks are copied straight into it while the next ones render) or pageable (a plain array:
 * chunks pass through pinned staging and are copied on by worker threads of the ctx; about 15 % slower). */
int tcrt_render(tcrt_ctx* ctx, const tcrt_params* params, float* host_rgb, tcrt_stats* stats);
/* Columns [x0,x1) only -> host_rgb_band[(x1-x0)*height*3].  This is what one rank of a
 * one-process-per-GPU launch calls for its band. */
int tcrt_render_columns(tcrt_ctx* ctx, const tcrt_params* params, int x0, int x1, float* host_rgb_band,
                        tcrt_stats* stats);
/* Same, result left in device memory (no copy-back); tcrt_download fetches it later. */
int tcrt_render_device(tcrt_ctx* ctx, const tcrt_params* params, int x0, int x1, tcrt_stats* stats);
int tcrt_download(tcrt_ctx* ctx, float* host_rgb_band);
/* Asynchronous frames (multi-frame mode, SURVEY §8f): tcrt_render_async queues columns [x0,x1) of a frame — into
 * host_rgb_band when it is not NULL, which should then be pinned (tcrt_alloc_host) — and returns at once with a
 * ticket; tcrt_wait(ticket) returns when that frame (and its copy-back) is complete and fills stats.  Every
 * device holds two frame buffers, so frame n+1 renders while frame n's band crosses the bus: at most two
 * frames are in flight, and a third tcrt_render_async fails with TCRT_ERR_INVALID until one has been waited
 * for.  tcrt_set_camera / tcrt_upload_scene between the calls apply to the frames queued after them.  The
 * "last render" the synchronous calls refer to (tcrt_download, tcrt_write_*) is the last frame WAITED for. */
int tcrt_render_async(tcrt_ctx* ctx, const tcrt_params* params, int x0, int x1, float* host_rgb_band, int* ticket);
int tcrt_wait(tcrt_ctx* ctx, int ticket, tcrt_stats* stats);
/* 8-bit frames: tcrt_render, tcrt_render_columns and tcrt_render_async with 3 bytes per pixel crossing the bus instead of
 * 12.  x-major like tcrt_render: byte (x*height + z)*3 + c, q(c) = floor(clamp(c,0,1)*255 + 0.5) (NaN -> 0), the
 * quantisation of tcrt_write_ppm; a column band is one contiguous slice.  Each column chunk is quantised on the device
 * by one more launch behind its render launch; the float frame stays on the device and remains "the last render" of
 * tcrt_download, tcrt_device_frame and the writers.  Pinned and pageable destinations as in tcrt_render.  A NULL
 * destination is TCRT_ERR_INVALID (the device-only call is tcrt_render_device).  RGB8 and float frames share tcrt_wait
 * and the two frames in flight.  Image rows (top row first) are the free view transpose(1,0,2)[::-1] of the array. */
int tcrt_render_rgb8(tcrt_ctx* ctx, const tcrt_params* params, unsigned char* host_rgb8, tcrt_stats* stats);
int tcrt_render_columns_rgb8(tcrt_ctx* ctx, const tcrt_params* params, int x0, int x1, unsigned char* host_rgb8_band,
                             tcrt_stats* stats);
int tcrt_render_async_rgb8(tcrt_ctx* ctx, const tcrt_params* params, int x0, int x1, unsigned char* host_rgb8_band,
                           int* ticket);
/* Supersampled (anti-aliased) frames: ss x ss samples per pixel, ss = samples per axis, 1 <= ss <= 8.  Sample (i, j),
 * 0 <= i, j < ss, of output pixel (x, z) is the reference's pixel (ss*x + i, ss*z + j) of the same scene, camera and
 * params at (ss*width, ss*height): every sample is a value the reference computes, so the grid is anchored at the
 * pixel's corner as the reference's rays are, and an ss > 1 image is shifted by (ss-1)/(2*ss) pixel against the ss = 1
 * image.  Resolve, in binary32, in exactly this order: acc = sample(0,0); acc += sample(i,j) for i = 0..ss-1 (outer),
 * j = 0..ss-1 (inner), skipping (0,0); out = acc / (float)(ss*ss) (IEEE division; no FMA, no pairwise tree; NaN and inf
 * propagate).  ss = 1 is the plain frame, bit for bit.  ss < 1: TCRT_ERR_INVALID; ss > 8, or ss*width or ss*height above
 * 2^24 (where (float)x stops being exact): TCRT_ERR_UNSUPPORTED, as is a frame whose column chunks would exceed the
 * kernels' index range (ss*ss*height*columns of a chunk above 2^31/3 sample channels).
 * The output is the W x H frame, x-major like tcrt_render, a column band [x0,x1) one contiguous slice; host_rgb_band NULL
 * leaves it on the device (tcrt_render_device).  The RGB8 forms carry quant8 of the resolved floats (not the mean of
 * quantised samples); their destination must not be NULL.  The resolved float frame becomes the last render of
 * tcrt_download, tcrt_device_frame and the writers.  Stats: rays_* count the rays of the whole sample frame,
 * col_begin/col_end are output columns, render_ms and gpu_launches include the resolve launches.  Pinned and pageable
 * destinations, multi-device contexts, tcrt_wait and the two frames in flight as in tcrt_render / tcrt_render_async. */
int tcrt_render_columns_ss(tcrt_ctx* ctx, const tcrt_params* params, int ss, int x0, int x1, float* host_rgb_band,
                           tcrt_stats* stats);
int tcrt_render_columns_ss_rgb8(tcrt_ctx* ctx, const tcrt_params* params, int ss, int x0, int x1,
                                unsigned char* host_rgb8_band, tcrt_stats* stats);
int tcrt_render_async_ss(tcrt_ctx* ctx, const tcrt_params* params, int ss, int x0, int x1, float* host_rgb_band,
                         int* ticket);
int tcrt_render_async_ss_rgb8(tcrt_ctx* ctx, const tcrt_params* params, int ss, int x0, int x1,
                              unsigned char* host_rgb8_band, int* ticket);
/* Adaptive anti-aliasing: the samples of tcrt_render_columns_ss traced only where the plain frame shows contrast.  For
 * params p (W x H), ss (1 <= ss <= 8) and contrast (-1 <= contrast <= 255):
 *   - P is the plain frame, exactly what tcrt_render returns for p; q(c) is the quant8 above;
 *   - pixel (x, z) is refined when contrast < 0, or when some neighbour (x', z') != (x, z) with |x'-x| <= 1 and
 *     |z'-z| <= 1 inside [0, W) x [0, H) has max over c of |q(P(x,z)_c) - q(P(x',z')_c)| > contrast.  Neighbours are
 *     taken from the frame, not from the requested band: a band's result does not depend on where the band is cut;
 *   - output pixel (x, z) is exactly the pixel of tcrt_render_columns_ss at the same ss where refined, exactly P(x, z)
 *     otherwise.  The RGB8 form carries quant8 of that float.
 * So contrast -1 gives the tcrt_render_columns_ss frame, contrast 255 and ss = 1 the plain frame (the mask is still
 * computed: an edge preview).  A refined pixel is resolved from the plain pixel, which is its sample (0,0) bit for bit
 * (the quotient x/W is the same at ss*W), and its ss*ss-1 other samples, in the order and arithmetic of
 * tcrt_render_columns_ss.
 * host_mask (may be NULL): one byte per pixel of the band, 1 refined / 0 not, x-major: host_mask[(x-x0)*H + z].
 * n_refined (may be NULL): the refined pixels of the band, over all devices.  host_rgb_band NULL leaves the frame on the
 * device (float form only; the RGB8 destination must not be NULL).  Pinned and pageable destinations as in tcrt_render.
 * Errors: ss < 1 or contrast outside [-1, 255]: TCRT_ERR_INVALID; ss > 8, or ss*W or ss*H above 2^24:
 * TCRT_ERR_UNSUPPORTED.  A long list of refined pixels is traced in pieces, never refused.
 * The call is synchronous: it renders the plain frame over the band and one halo column each side, classifies and
 * compacts the band on the device, reads the list's length (4 bytes), then traces and resolves the list's samples.  The
 * resolved frame becomes the last render (tcrt_download, tcrt_device_frame, the writers); with frames in flight the
 * rules of tcrt_render_columns_ss apply.  A multi-device ctx renders bands of equal width and neither reads nor updates
 * the balanced cut or its cost map.  Stats: col_begin/col_end per device; render_ms from the first launch to the last
 * (it includes the wait for the list's length); gpu_launches every launch; rays_* every ray traced, rays_primary =
 * (band + halo columns)*H + (ss*ss-1)*n_refined. */
int tcrt_render_columns_adaptive(tcrt_ctx* ctx, const tcrt_params* params, int ss, int contrast, int x0, int x1,
                                 float* host_rgb_band, unsigned char* host_mask, unsigned long long* n_refined,
                                 tcrt_stats* stats);
int tcrt_render_columns_adaptive_rgb8(tcrt_ctx* ctx, const tcrt_params* params, int ss, int contrast, int x0, int x1,
                                      unsigned char* host_rgb8_band, unsigned char* host_mask,
                                      unsigned long long* n_refined, tcrt_stats* stats);
/* Device address of a device's band of the last render (for zero-copy consumers, e.g. a
 * torch tensor view); floats = (col_end-col_begin)*height*3. */
int tcrt_device_frame(tcrt_ctx* ctx, int device_slot, void** dev_ptr, size_t* n_floats);
/* Primary-hit buffers: what is at each pixel.  For pixel (x, z) of the params.width x params.height frame:
 *   - primary ray: the ray the render traces (Camera::createEyeRay at x / W, z / H);
 *   - nearest hit: the reference's getCollision (RayTracer.cpp:50-89), lexicographic on (distance, object index); hits at
 *     or beyond far_dist are invisible; lights are objects like any other;
 *   - object (int32): the object index of the nearest hit (its position in the scene's list, as in tcrt_scene), -1 on
 *     a miss;
 *   - distance (float32): the winning primitive's distance exactly as the reference computes it; negative when the eye
 *     is inside a sphere (SceneSphere.cpp:139); far_dist on a miss;
 *   - normal (3 x float32): the direction of the hit's normal ray (CollisionObject, SceneObject.h:47-105): the
 *     primitive's normal re-normalised by Ray(point, normal), for planes the side facing the ray (computeNormal);
 *     (+0, +0, +0) on a miss.
 * The result does not depend on max_depth, shadows_on, reflections_on or null_color.  Layout x-major like frames:
 * object[(x-x0)*H + z], distance[(x-x0)*H + z], normal[((x-x0)*H + z)*3 + c]; a column band is one contiguous slice of
 * each buffer.  Supersampled hit buffers do not exist.
 *
 * tcrt_hit_buffers: columns [x0, x1).  All three buffers are computed on the device (20 B per pixel); a NULL host pointer
 * is not copied back, all three NULL leaves them on the device only (tcrt_device_hit_buffers).  Pinned and pageable
 * destinations as in tcrt_render.  A multi-device ctx computes one band of equal width per device.  Stats: col_begin /
 * col_end per device, render_ms = kernel time, d2h_ms as for frames, rays_primary = pixels, no shadow or reflection
 * rays, gpu_launches = kernel launches.  Errors as for frames.
 * tcrt_device_hit_buffers: device addresses of a device's band of the last tcrt_hit_buffers call, n_pixels per buffer
 * (normal holds 3 * n_pixels floats); TCRT_ERR_NO_FRAME before the first call.
 * tcrt_pick: the hits of n pixels xz[2i] = x, xz[2i+1] = z on device slot 0, into object[i], distance[i],
 * normal[3i..3i+2]; each output pointer may be NULL.  n = 0 launches nothing.  A pixel outside the frame is
 * TCRT_ERR_INVALID and nothing is written.
 * None of these calls changes the last render (tcrt_download, tcrt_device_frame, the writers), the multi-device cut or
 * cost map, or a frame in flight: they have buffers of their own, may be called while two frames are in flight and do
 * not count as one.  They trace with the camera of tcrt_set_camera, like frames. */
int tcrt_hit_buffers(tcrt_ctx* ctx, const tcrt_params* params, int x0, int x1, int* host_object, float* host_distance,
                     float* host_normal, tcrt_stats* stats);
int tcrt_device_hit_buffers(tcrt_ctx* ctx, int device_slot, int** object, float** distance, float** normal,
                            size_t* n_pixels);
int tcrt_pick(tcrt_ctx* ctx, const tcrt_params* params, int n, const int* xz, int* object, float* distance,
              float* normal);
/* Ray batches: what caller-supplied rays see, and what they hit.  A batch is n rays; ray i has origin o_i =
 * origins[3i..3i+2] (or origins[0..2] for every ray when shared_origin != 0) and direction d_i = directions[3i..3i+2],
 * all float32.
 *   - colour (tcrt_trace_rays): rgb[3i..3i+2] is what the reference's calculatePixel returns at level 0 for a Ray whose
 *     stored origin and direction are exactly o_i and d_i, with the uploaded scene and params max_depth, shadows_on,
 *     reflections_on, null_color and far_dist.  width, height and the camera are not read;
 *   - nearest hit (tcrt_intersect_rays): object[i], distance[i], normal[3i..3i+2] with the definitions of
 *     tcrt_hit_buffers applied to ray i (object index or -1; the reference's distance, negative inside a sphere, far_dist
 *     on a miss; n2, or (+0, +0, +0) on a miss).  Only far_dist is read.  Any output pointer may be NULL, not all three.
 * Directions are used as given, not normalised again: a Ray stores the direction its constructor has normalised, and
 * vector3d::normalize is not idempotent to the bit.  A caller with raw directions (x, y, z) applies the reference's
 * normalisation: len = sqrtf((x*x + y*y) + z*z), then x/len, y/len, z/len (binary32, no FMA, IEEE division and square root).
 * A ray is traced only when it is valid: all six components finite, |o_k| <= 2^40, and s = (dx*dx + dy*dy) + dz*dz in
 * binary32 without FMA satisfies |s - 1| <= 2^-21.  Every direction that normalisation makes of a vector whose squared
 * length is a normal float passes (DESIGN.md 4.5).  An invalid ray is not traced and not counted as a ray: its colour
 * is quiet NaN (0x7fc00000) in all three channels; its hit is object -2, distance NaN, normal NaN.  *n_invalid (may be
 * NULL) returns their number; the call still succeeds.  The check runs on the device, in the kernel that traces the batch.
 * A warp takes 32 consecutive rays: rays that are close in the batch should be close in space (e.g. 4 x 8 pixel tiles
 * of a camera), or the walks of a warp diverge and the batch is slower (profiles/README.md 12).  The library does not sort.
 * Host forms: inputs and outputs in pinned or pageable memory (identical results).  A multi-device ctx splits [0, n) into
 * equal contiguous ranges, one per device.  The batch runs in pieces of at most 4 Mi rays round robin over the render
 * streams: each piece's inputs are copied in (24 B per ray, 12 with a shared origin), traced by one launch, and its
 * outputs copied out while later pieces trace.
 * Device forms (_device): one device slot; every pointer must be device memory of that device (cudaPointerGetAttributes),
 * else TCRT_ERR_INVALID; the caller has finished writing the inputs (e.g. synchronised its stream).
 * All four calls are synchronous.  n = 0 launches nothing.  Errors: NULL ctx, params, inputs (n > 0) or outputs, or n
 * whose byte count overflows: TCRT_ERR_INVALID; tcrt_trace_rays* with max_depth < 0: TCRT_ERR_INVALID, above
 * TCRT_MAX_DEPTH: TCRT_ERR_UNSUPPORTED; before tcrt_upload_scene: TCRT_ERR_NO_SCENE.
 * Stats: col_begin/col_end are each device's ray range [begin, end) (clipped to INT_MAX), rays_primary the valid rays,
 * rays_shadow / rays_reflect as for frames (hits: 0), render_ms from the first input copy to the end of the last launch,
 * d2h_ms the copy-back time not hidden behind the launches, gpu_launches the launches.
 * Like hit buffers, these calls have buffers, queue heads and events of their own: they never change the last render,
 * the multi-device cut or cost map, or a frame in flight, may run while two frames are in flight and do not count as one.
 * tcrt_set_camera has no effect on them. */
int tcrt_trace_rays(tcrt_ctx* ctx, const tcrt_params* params, size_t n, const float* origins, int shared_origin,
                    const float* directions, float* rgb, unsigned long long* n_invalid, tcrt_stats* stats);
int tcrt_intersect_rays(tcrt_ctx* ctx, const tcrt_params* params, size_t n, const float* origins, int shared_origin,
                        const float* directions, int* object, float* distance, float* normal,
                        unsigned long long* n_invalid, tcrt_stats* stats);
int tcrt_trace_rays_device(tcrt_ctx* ctx, int device_slot, const tcrt_params* params, size_t n, const float* origins,
                           int shared_origin, const float* directions, float* rgb, unsigned long long* n_invalid,
                           tcrt_stats* stats);
int tcrt_intersect_rays_device(tcrt_ctx* ctx, int device_slot, const tcrt_params* params, size_t n,
                               const float* origins, int shared_origin, const float* directions, int* object,
                               float* distance, float* normal, unsigned long long* n_invalid, tcrt_stats* stats);
/* Occlusion queries: the reference's shadow test (inShadeCollisionDetection, RayTracer.cpp:709-739) for caller-supplied
 * rays, and its inShade (:743-771) for caller-supplied points against every light.  Neither takes tcrt_params: the shadow
 * test reads none of them (not far_dist, shadows_on or max_depth).
 *   - rays (tcrt_occluded_rays): origins and directions as for the ray batches above (per ray or shared origin, used as a
 *     Ray stores them, the same validity rule), plus a limit tmax[i] per ray.  occluded[i] = 1 when some object that is
 *     not a light has a reference collision at distance d < tmax_i (strict), else 0.  tmax = +inf is allowed.  A sphere's
 *     distance is negative when the origin is inside it, so an origin inside a non-light sphere is always occluded.
 *   - points (tcrt_occluded_lights): points[3i..3i+2], n points; occluded[i * n_lights + l] for every light l in the order
 *     of tcrt_scene.light_obj (increasing object index).  The value is what inShade(P_i, light l) returns, with the
 *     reference's arithmetic: dir = L - P, dist = sqrtf((dx*dx + dy*dy) + dz*dz), lr = dir / dist (three IEEE
 *     divisions), then the test above along lr with limit dist.  A scene without lights is success: nothing is written.
 * An answer of 0xFF marks an invalid ray or pair, which is not traced: a ray that fails the batch rule, or whose tmax is
 * NaN or <= 0; a pair whose point fails the origin rule (finite, |p_k| <= 2^40; the point's whole row), or whose lr fails
 * the direction rule (|s - 1| <= 2^-21).  The latter happens only when P is at the light or within about 1e-19 of it,
 * where the reference would answer "not in shade" (its 0/0 compares false); like the ray batches' rule, this is a
 * deliberate deviation.  *n_invalid (may be NULL) counts invalid rays, or invalid (point, light) pairs.
 * Host forms: inputs and outputs in pinned or pageable memory.  A multi-device ctx splits [0, n) into equal contiguous
 * ranges of rays or points.  Pieces of at most 4 Mi rays (28 B of input each, 16 with a shared origin) or 4 Mi (point,
 * light) pairs (12 B of input per point, n_lights bytes of output), at least one point, round robin over the render
 * streams.  Device forms (_device) as for the ray batches.  All four calls are synchronous; n = 0 launches nothing.
 * Errors: NULL ctx, inputs (n > 0) or output, or a byte count that overflows: TCRT_ERR_INVALID; before tcrt_upload_scene:
 * TCRT_ERR_NO_SCENE.  Stats: col_begin/col_end each device's range of rays or points, rays_shadow the tests traced (valid
 * rays or valid pairs), rays_primary and rays_reflect 0, render_ms, d2h_ms and gpu_launches as for the ray batches.  They
 * never change the last render, the writers, the multi-device cut or cost map, or a frame in flight, and ignore
 * tcrt_set_camera. */
int tcrt_occluded_rays(tcrt_ctx* ctx, size_t n, const float* origins, int shared_origin, const float* directions,
                       const float* tmax, unsigned char* occluded, unsigned long long* n_invalid, tcrt_stats* stats);
int tcrt_occluded_lights(tcrt_ctx* ctx, size_t n, const float* points, unsigned char* occluded,
                         unsigned long long* n_invalid, tcrt_stats* stats);
int tcrt_occluded_rays_device(tcrt_ctx* ctx, int device_slot, size_t n, const float* origins, int shared_origin,
                              const float* directions, const float* tmax, unsigned char* occluded,
                              unsigned long long* n_invalid, tcrt_stats* stats);
int tcrt_occluded_lights_device(tcrt_ctx* ctx, int device_slot, size_t n, const float* points, unsigned char* occluded,
                                unsigned long long* n_invalid, tcrt_stats* stats);
/* Cost-balanced column bands (replaces the equal z-bands of the reference's strategy 1,
 * RayTracer.cpp:904-906, whose load imbalance strategies 2-7 and PixelQueue were written to fix).
 * Renders a low-resolution copy of the frame on device slot 0 in which every finished pixel adds its
 * bounce count (reflection levels traced + 1) to its column and its row, then cuts [0, width) into
 * n_bands bands of equal estimated cost: bounds[0] = 0 <= bounds[1] <= ... <= bounds[n_bands] = width.
 * The estimate is deterministic for a (scene, camera, params); bounce counts are a proxy for time, so a
 * multi-process run computes the cut on one rank, shares it, and refines it from measured band times
 * (tcrt_rebalance_columns); a multi-device ctx computes it once per (scene, params). */
int tcrt_balance_columns(tcrt_ctx* ctx, const tcrt_params* params, int n_bands, int* bounds);
/* The cut itself (host only, no device needed): costs[i] >= 0 for n_costs equal-width column groups
 * covering [0, width).  When width is a multiple of 4 (and bands are at least 16 columns wide on
 * average) so is every cut: the kernel's pixel tiles are 4 columns wide. */
int tcrt_bands_from_costs(const double* costs, int n_costs, int width, int n_bands, int* bounds);

/* Feedback step (host only): given the kernel time ms[b] of every band of the cut `bounds`, the cut
 * that would equalise the times if cost were spread evenly inside each band.  Applied to consecutive
 * frames it converges on the measured balance (the role of the reference's self-scheduling
 * strategies 2/3, RayTracer.cpp:956-1079, between whole GPUs).  A multi-device ctx applies it after
 * every whole-frame render; bench.py applies it during warm-up. */
int tcrt_rebalance_columns(const int* bounds, const double* ms, int n_bands, int width, int* new_bounds);

/* Overwrite the L2 cache of every device of the ctx (benchmark hygiene between timed steps). */
int tcrt_flush_l2(tcrt_ctx* ctx);
/* FP32-pipe microbenchmark on device slot 0 (the roofline denominator of this path, SURVEY
 * §8d): sustained lane-operations per second of dependent-chain FMUL+FADD pairs (unfused, the
 * instruction mix parity-exact code issues) and of FFMA, in units of 1e12 lane-instructions/s,
 * plus the kernel time of each probe.  FFMA counts 1 instruction (2 flops). */
int tcrt_fp32_peak(tcrt_ctx* ctx, double* unfused_tera_inst, double* fma_tera_inst, double* ms_each);

/* ---- beyond the reference (SURVEY §8f) ------------------------------------------------------------ */
/* Multi-frame mode: replaces the camera of the uploaded scene without touching the scene (the
 * reference renders one static frame and lists moving scenes as unsupported, README.md:29).  The
 * camera travels with every launch, so this is free; the next render uses it. */
int tcrt_set_camera(tcrt_ctx* ctx, const tcrt_camera* camera);
/* The last render as a binary PPM (P6, 8 bits per channel, q(c) = floor(clamp(c,0,1)*255 + 0.5)),
 * viewable directly: image column = x, image row 0 = the TOP (z = height-1), as the reference's
 * offline viewer would show the .txt.  Quantised on the GPU, 3 B/pixel cross the bus. */
int tcrt_write_ppm(tcrt_ctx* ctx, const tcrt_params* params, const char* path);
/* The last render as raw little-endian float32 (the binary output the reference leaves as a TODO,
 * RayTracer.cpp:1605-1613): a 32-byte header "TCRTBIN1" + int32 width, height + 16 zero bytes, then
 * width*height*3 floats in the order of pixels[W][H] (x-major, z fastest, r g b). */
int tcrt_write_bin(tcrt_ctx* ctx, const tcrt_params* params, const char* path);

/* Self-test on device slot 0: the render kernel's shared-reciprocal division (three quotients by one
 * length, used for vector3d::normalize, vector3d.h:57-74) against the IEEE division instruction
 * sequence on n_cases pseudo-random operand triples; *n_bad = cases with any differing bit. */
int tcrt_selftest_div3(tcrt_ctx* ctx, unsigned long long n_cases, unsigned int seed, unsigned long long* n_bad);

/* ---- .txt writer (replaces init_log + printPixelsToLog) --------------------------- */
/* Bytes of the pixel lines "(%f, %f, %f)\n" of the last render (all its columns). */
int tcrt_txt_size(tcrt_ctx* ctx, size_t* n_bytes);
/* Formats the last render's pixel lines on the GPU and copies them to host_text (capacity
 * cap bytes, no terminator); *n_bytes = length.  Byte-identical to glibc's
 * sprintf("(%f, %f, %f)\n") of the same floats (RayTracer.cpp:1601). */
int tcrt_format_txt(tcrt_ctx* ctx, char* host_text, size_t cap, size_t* n_bytes);
/* Same formatter applied to caller-supplied pixels (n_pixels*3 floats in host memory): H2D,
 * format on device 0 of the ctx, D2H.  Independent of the last render (the reference's
 * main_test, RayTracer.cpp:1412-1444, drives its writer this way). */
int tcrt_format_pixels(tcrt_ctx* ctx, const float* host_rgb, size_t n_pixels, char* host_text, size_t cap,
                       size_t* n_bytes);
/* Header lines of the file (init_log RayTracer.cpp:2033-2058 + the three tag lines of
 * printPixelsToLog :1576-1578), x86 personality: "OSX Awesome Picture", Hardware_Target
 * "OSX C++", Number_of_Cores 1, IS_FOR_HARDWARE, NO_PARTIONING.  Returns length written
 * (excluding the terminating NUL) or a negative error. */
int tcrt_txt_header(const tcrt_params* params, double run_time_s, char* buf, size_t cap);
/* Whole file: header + pixel lines of the last render (must have covered columns
 * [0,width)).  run_time_s feeds the Run_Time / us/pixel tags. */
int tcrt_write_txt(tcrt_ctx* ctx, const tcrt_params* params, const char* path, double run_time_s);
/* One file from several processes (one per GPU, each holding one band of columns): one process creates the
 * file — header + room for width*height lines of 31 bytes, the length of every pixel line whose channels
 * are in [0, 10) — and, after a barrier of the caller's, every process writes the lines of the band it last
 * rendered at their place (x-major order makes a band one run of lines, so no band waits for another).
 * TCRT_ERR_UNSUPPORTED if a line of the band is not 31 bytes: gather the bands and use tcrt_write_txt.
 * run_time_s must be the same in all calls (it is part of the header, whose length positions the lines). */
int tcrt_txt_create(const tcrt_params* params, const char* path, double run_time_s);
int tcrt_write_txt_band(tcrt_ctx* ctx, const tcrt_params* params, const char* path, double run_time_s);

#ifdef __cplusplus
}
#endif
#endif /* TCRT_H_ */
