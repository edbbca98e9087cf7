// include/RayTracer.h — C++ convenience over the C ABI (include/tcrt.h), shaped like the
// reference's driver: raytrace_main() (RayTracer.cpp:855-1114) = build scene, render every
// pixel, printPixelsToLog().  Header-only; link with libtcrt.so.
#ifndef TCRT_RAYTRACER_H_
#define TCRT_RAYTRACER_H_

#include <chrono>
#include <string>
#include <vector>

#include "CelioRayTracer.hpp"
#include "tcrt.h"

#define LOG_FILE_NAME "raytracer_screen.txt"   // RayTracer.h:134

namespace CelioRayTracer {

// The compile-time knobs of rt_project_parameters.h, at run time.
struct RenderSettings {
    int width = 500;          // SCREEN_HORIZONTAL_RESOLUTION
    int height = 504;         // SCREEN_VERTICAL_RESOLUTION
    int max_depth = 50;       // MAX_RECURSION_LEVEL
    bool shadows = true;      // SHADOWS_ON
    bool reflections = true;  // REFLECTIONS_ON
    int samples = 1;          // samples per axis: > 1 renders the anti-aliased frame of tcrt_render_columns_ss
    int contrast = -1;        // with samples > 1: >= 0 supersamples only the pixels at quant8 contrast edges above this
                              // (tcrt_render_columns_adaptive); -1 supersamples every pixel
    tcrt_params params() const {
        tcrt_params p;
        tcrt_default_params(&p);
        p.width = width; p.height = height; p.max_depth = max_depth;
        p.shadows_on = shadows; p.reflections_on = reflections;
        return p;
    }
};

// Owns a tcrt_ctx on one or more B200s.
class GpuRayTracer {
public:
    explicit GpuRayTracer(const std::vector<int>& devices = std::vector<int>(1, 0)) : ctx_(NULL), run_time_s_(0) {
        rc_ = tcrt_create(&ctx_, devices.data(), (int)devices.size());
    }
    ~GpuRayTracer() { tcrt_destroy(ctx_); }
    bool ok() const { return rc_ == TCRT_OK; }
    const char* lastError() const { return tcrt_last_error(ctx_); }

    // my_scene / my_camera of the reference (RayTracer.h:50-51) become resident device data
    int setScene(const Scene& scene, const Camera& camera) {
        scene.flatten(flat_);
        tcrt_scene s = flat_.view();
        tcrt_camera c;
        camera.exportTo(&c);
        return rc_ = tcrt_upload_scene(ctx_, &s, &c);
    }
    // moving spheres (tcrt_update_spheres): geom[4*i .. 4*i+3] = centre xyz and radius*radius of sphere i, in the order of
    // the scene given to setScene; the scene stays resident, the GPU refits its structures
    int updateSpheres(const float* geom, tcrt_stats* stats = NULL) { return rc_ = tcrt_update_spheres(ctx_, geom, stats); }
    // material edits (tcrt_update_materials, tcrt_update_textures): `scene` is the scene given to setScene, edited with the
    // ObjMaterial / SceneObject setters; the colour, factors, intensity and texture id of objects[0 .. n) and every checker
    // row are sent.  A scene whose counts, lights or number of textures differ from the uploaded one: TCRT_ERR_INVALID
    // (that takes setScene).  stats: of the objects' rows.
    int updateMaterials(const Scene& scene, const int* objects, int n, tcrt_stats* stats = NULL) {
        SceneFlattener f;
        scene.flatten(f);
        if (f.n_objects != flat_.n_objects || f.sphere_obj.size() != flat_.sphere_obj.size() ||
            f.fin_obj.size() != flat_.fin_obj.size() || f.inf_obj.size() != flat_.inf_obj.size() ||
            f.light_obj != flat_.light_obj || f.textures.size() != flat_.textures.size() || n < 0 || (n > 0 && !objects))
            return rc_ = TCRT_ERR_INVALID;
        std::vector<float> surface(4 * (size_t)n), material(4 * (size_t)n);
        std::vector<int> texture(n);
        for (int i = 0; i < n; i++) {
            const int o = objects[i];
            if (o < 0 || o >= f.n_objects) return rc_ = TCRT_ERR_INVALID;
            for (int k = 0; k < 4; k++) {
                surface[4 * i + k] = f.obj_surface[4 * o + k];
                material[4 * i + k] = f.obj_material[4 * o + k];
            }
            texture[i] = f.obj_info[4 * o + 3];
        }
        if (n > 0 && (rc_ = tcrt_update_materials(ctx_, n, objects, surface.data(), material.data(), texture.data(), stats)))
            return rc_;
        std::vector<int> ids(f.textures.size() / 8);
        for (size_t t = 0; t < ids.size(); t++) ids[t] = (int)t;
        return rc_ = ids.empty() ? TCRT_OK : tcrt_update_textures(ctx_, (int)ids.size(), ids.data(), f.textures.data(), NULL);
    }
    // moving planes (tcrt_update_planes): `moved` is a scene built in the object order of the scene given to setScene, with
    // some planes constructed elsewhere; the geometry, normals and origin of objects[0 .. n) are sent.  A scene whose
    // counts, object types or lights differ from the uploaded one, or an object that is not a plane: TCRT_ERR_INVALID
    // (that takes setScene).
    int updatePlanes(const Scene& moved, const int* objects, int n, tcrt_stats* stats = NULL) {
        SceneFlattener f;
        moved.flatten(f);
        if (f.n_objects != flat_.n_objects || f.sphere_obj.size() != flat_.sphere_obj.size() ||
            f.fin_obj.size() != flat_.fin_obj.size() || f.inf_obj.size() != flat_.inf_obj.size() ||
            f.light_obj != flat_.light_obj || n < 0 || (n > 0 && !objects))
            return rc_ = TCRT_ERR_INVALID;
        for (int o = 0; o < f.n_objects; o++)
            if (f.obj_info[4 * o] != flat_.obj_info[4 * o]) return rc_ = TCRT_ERR_INVALID;
        std::vector<float> geom(16 * (size_t)n), normals(8 * (size_t)n), origin(4 * (size_t)n);
        for (int i = 0; i < n; i++) {
            const int o = objects[i];
            if (o < 0 || o >= f.n_objects || f.obj_info[4 * o] == TCRT_SPHERE) return rc_ = TCRT_ERR_INVALID;
            const std::vector<float>& rows = f.obj_info[4 * o] == TCRT_FINITE_PLANE ? f.fin_geom : f.inf_geom;
            for (int k = 0; k < 16; k++) geom[16 * i + k] = rows[16 * (size_t)f.obj_info[4 * o + 1] + k];
            for (int k = 0; k < 8; k++) normals[8 * i + k] = f.obj_normals[8 * (size_t)o + k];
            for (int k = 0; k < 4; k++) origin[4 * i + k] = f.obj_origin[4 * (size_t)o + k];
        }
        return rc_ = tcrt_update_planes(ctx_, n, objects, geom.data(), normals.data(), origin.data(), stats);
    }
    // the pixel loop (RayTracer.cpp:911-923): pixels[x][z] -> pixels_xmajor[(x*H + z)*3 + c]; with rs.samples > 1 each
    // pixel is the mean of rs.samples x rs.samples samples (tcrt_render_columns_ss), with rs.contrast >= 0 only the pixels
    // at contrast edges (tcrt_render_columns_adaptive)
    int render(const RenderSettings& rs, float* pixels_xmajor, tcrt_stats* stats = NULL) {
        settings_ = rs;
        tcrt_params p = rs.params();
        std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
        if (rs.samples != 1 && rs.contrast >= 0)
            rc_ = tcrt_render_columns_adaptive(ctx_, &p, rs.samples, rs.contrast, 0, p.width, pixels_xmajor, NULL, NULL, stats);
        else if (rs.samples != 1)
            rc_ = tcrt_render_columns_ss(ctx_, &p, rs.samples, 0, p.width, pixels_xmajor, stats);
        else
            rc_ = pixels_xmajor ? tcrt_render(ctx_, &p, pixels_xmajor, stats)
                                : tcrt_render_device(ctx_, &p, 0, p.width, stats);
        run_time_s_ = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        return rc_;
    }
    // the same frame quantised to 8 bits on the GPU: pixels_xmajor_rgb8[(x*H + z)*3 + c] = floor(clamp(c,0,1)*255 + 0.5);
    // the float frame stays the last render (printPixelsToLog writes it); rs.samples > 1: of the anti-aliased frame
    int renderRGB8(const RenderSettings& rs, unsigned char* pixels_xmajor_rgb8, tcrt_stats* stats = NULL) {
        settings_ = rs;
        tcrt_params p = rs.params();
        std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
        if (rs.samples != 1 && rs.contrast >= 0)
            rc_ = tcrt_render_columns_adaptive_rgb8(ctx_, &p, rs.samples, rs.contrast, 0, p.width, pixels_xmajor_rgb8, NULL,
                                                    NULL, stats);
        else
            rc_ = rs.samples != 1 ? tcrt_render_columns_ss_rgb8(ctx_, &p, rs.samples, 0, p.width, pixels_xmajor_rgb8, stats)
                                  : tcrt_render_rgb8(ctx_, &p, pixels_xmajor_rgb8, stats);
        run_time_s_ = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        return rc_;
    }
    // what is at each pixel of the frame rs describes (tcrt_hit_buffers), x-major like render: obj[x*H + z] the object
    // index of the primary ray's nearest hit (-1: miss), dist[x*H + z] its distance, normal[(x*H + z)*3 + c] its normal;
    // a NULL pointer is not copied back.  The last render is not touched.  Not for rs.samples != 1.
    int hitBuffers(const RenderSettings& rs, int* obj, float* dist, float* normal, tcrt_stats* stats = NULL) {
        if (rs.samples != 1) return rc_ = TCRT_ERR_UNSUPPORTED;
        tcrt_params p = rs.params();
        return rc_ = tcrt_hit_buffers(ctx_, &p, 0, p.width, obj, dist, normal, stats);
    }
    // the object under pixel (x, z) (tcrt_pick), its distance and normal (3 floats); any pointer may be NULL
    int pick(const RenderSettings& rs, int x, int z, int* obj, float* dist = NULL, float* normal3 = NULL) {
        if (rs.samples != 1) return rc_ = TCRT_ERR_UNSUPPORTED;
        tcrt_params p = rs.params();
        const int xz[2] = {x, z};
        return rc_ = tcrt_pick(ctx_, &p, 1, xz, obj, dist, normal3);
    }
    // what each ray sees (tcrt_trace_rays): rgb[3i..3i+2] is calculatePixel of rays[i] at level 0, with rs's depth and
    // switches; the rays are traced with the origin and direction they hold (built by Camera::createEyeRay or Ray(o, d),
    // which normalise), so rays[i] gives what the reference computes for it.  An invalid ray (tcrt.h) gets NaN.
    int traceRays(const RenderSettings& rs, const std::vector<Ray>& rays, float* rgb, unsigned long long* n_invalid = NULL,
                  tcrt_stats* stats = NULL) {
        std::vector<float> o, d;
        unpackRays(rays, o, d);
        tcrt_params p = rs.params();
        return rc_ = tcrt_trace_rays(ctx_, &p, rays.size(), o.data(), 0, d.data(), rgb, n_invalid, stats);
    }
    // the nearest hits of the rays (tcrt_intersect_rays): obj[i], dist[i], normal[3i..3i+2] as hitBuffers defines them
    // (object -2 for an invalid ray); any pointer may be NULL, not all three
    int intersectRays(const RenderSettings& rs, const std::vector<Ray>& rays, int* obj, float* dist, float* normal,
                      unsigned long long* n_invalid = NULL, tcrt_stats* stats = NULL) {
        std::vector<float> o, d;
        unpackRays(rays, o, d);
        tcrt_params p = rs.params();
        return rc_ = tcrt_intersect_rays(ctx_, &p, rays.size(), o.data(), 0, d.data(), obj, dist, normal, n_invalid, stats);
    }
    // inShadeCollisionDetection(rays[i], tmax[i]) (tcrt_occluded_rays): occluded[i] = 1 when a non-light object is hit
    // nearer than tmax[i], else 0; 0xFF for an invalid ray or tmax (tcrt.h).  tmax.size() must equal rays.size().
    int occludedRays(const std::vector<Ray>& rays, const std::vector<float>& tmax, unsigned char* occluded,
                     unsigned long long* n_invalid = NULL, tcrt_stats* stats = NULL) {
        if (tmax.size() != rays.size()) return rc_ = TCRT_ERR_INVALID;
        std::vector<float> o, d;
        unpackRays(rays, o, d);
        return rc_ = tcrt_occluded_rays(ctx_, rays.size(), o.data(), 0, d.data(), tmax.data(), occluded, n_invalid, stats);
    }
    // inShade(points[i], light l) for every light (tcrt_occluded_lights): occluded[i * n_lights + l], lights in increasing
    // object index; 0xFF for an invalid pair (tcrt.h)
    int occludedLights(const std::vector<vector3d>& points, unsigned char* occluded, unsigned long long* n_invalid = NULL,
                       tcrt_stats* stats = NULL) {
        std::vector<float> p(points.size() * 3);
        for (size_t i = 0; i < points.size(); i++) {
            p[3 * i] = points[i].x; p[3 * i + 1] = points[i].y; p[3 * i + 2] = points[i].z;
        }
        return rc_ = tcrt_occluded_lights(ctx_, points.size(), p.data(), occluded, n_invalid, stats);
    }
    // the scene from every camera of `cameras` in one call (tcrt_render_views): view v is exactly render(rs, ...) after
    // the scene's camera is set to cameras[v], stacked view-major, rgb[((v*W + x)*H + z)*3 + c]; rgb8 (may be NULL, and
    // rgb may be NULL when it is not) the same quantised to 8 bits.  The last render and the scene's camera are not
    // touched.  Not for rs.samples != 1.
    int renderViews(const RenderSettings& rs, const std::vector<Camera>& cameras, float* rgb, unsigned char* rgb8 = NULL,
                    tcrt_stats* stats = NULL) {
        if (rs.samples != 1) return rc_ = TCRT_ERR_UNSUPPORTED;
        std::vector<tcrt_camera> c(cameras.size());
        for (size_t i = 0; i < cameras.size(); i++) cameras[i].exportTo(&c[i]);
        tcrt_params p = rs.params();
        return rc_ = tcrt_render_views(ctx_, &p, (int)cameras.size(), c.data(), rgb, rgb8, stats);
    }
    // init_log + printPixelsToLog (RayTracer.cpp:2022-2061,1574-1626)
    int printPixelsToLog(const char* path = LOG_FILE_NAME) {
        tcrt_params p = settings_.params();
        return rc_ = tcrt_write_txt(ctx_, &p, path, run_time_s_);
    }
    double runTimeSeconds() const { return run_time_s_; }
    tcrt_ctx* handle() { return ctx_; }

private:
    static void unpackRays(const std::vector<Ray>& rays, std::vector<float>& o, std::vector<float>& d) {
        o.resize(rays.size() * 3);
        d.resize(rays.size() * 3);
        for (size_t i = 0; i < rays.size(); i++) {
            const vector3d ro = rays[i].getOrigin(), rd = rays[i].getDirection();
            o[3 * i] = ro.x; o[3 * i + 1] = ro.y; o[3 * i + 2] = ro.z;
            d[3 * i] = rd.x; d[3 * i + 1] = rd.y; d[3 * i + 2] = rd.z;
        }
    }
    tcrt_ctx* ctx_;
    int rc_;
    double run_time_s_;
    RenderSettings settings_;
    SceneFlattener flat_;
};

// raytrace_main (RayTracer.cpp:855): 0 ok, 1 error, like the reference.
inline int raytrace_main(const Scene& scene, const Camera& camera, const RenderSettings& rs = RenderSettings(),
                         const char* log_path = LOG_FILE_NAME, const std::vector<int>& devices = std::vector<int>(1, 0)) {
    GpuRayTracer rt(devices);
    if (!rt.ok()) { fprintf(stderr, "%s\n", rt.lastError()); return 1; }
    if (rt.setScene(scene, camera) || rt.render(rs, NULL) || rt.printPixelsToLog(log_path)) {
        fprintf(stderr, "%s\n", rt.lastError());
        return 1;
    }
    return 0;
}

}  // namespace CelioRayTracer
#endif  // TCRT_RAYTRACER_H_
