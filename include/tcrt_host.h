/* include/tcrt_host.h — C binding of the host construction API (include/CelioRayTracer.hpp)
 * for callers that cannot include C++ headers (ctypes in tests/ and bench.py, other FFIs).
 * Each function is a one-line forward to the C++ method named in its comment; semantics,
 * argument order and defaults are those of the reference's public API (SURVEY.md §8b).
 * Handles are opaque; objects are owned by their scene once added.  Part of libtcrt.so.
 */
#ifndef TCRT_HOST_H_
#define TCRT_HOST_H_

#include "tcrt.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tcrt_hscene tcrt_hscene;   /* CelioRayTracer::Scene + its flattened form */
typedef struct tcrt_hcamera tcrt_hcamera; /* CelioRayTracer::Camera */

tcrt_hscene* tcrt_hscene_new(void);                                /* Scene::Scene() */
void tcrt_hscene_free(tcrt_hscene* s);
tcrt_hcamera* tcrt_hcamera_new(void);                              /* Camera::Camera() */
void tcrt_hcamera_free(tcrt_hcamera* c);
void tcrt_hcamera_set_two_mirrors(tcrt_hcamera* c);                /* Camera::setSceneTwoMirrors() */
/* Camera::aim: the reference's pose arithmetic (Camera.cpp:22-38) for the screen centre screen_origin3, the screen's x
 * axis horizontal3 and the viewing direction outwards3 (neither need be normalised): vertical = horizontal x outwards,
 * then all three normalised, the eye one unit behind the screen.  The screen size is kept. */
void tcrt_hcamera_aim(tcrt_hcamera* c, const float* screen_origin3, const float* horizontal3, const float* outwards3);
void tcrt_hcamera_export(const tcrt_hcamera* c, tcrt_camera* out);
/* Camera::createEyeRay(dx, dy): origin and normalised direction */
void tcrt_hcamera_eye_ray(const tcrt_hcamera* c, float dx_percent, float dy_percent, float* origin3, float* dir3);

/* Named scenes: "default" (Scene::initialize), "two_mirrors" (Scene::initializeTwoMirrors,
 * also re-aims the camera), "synth1024", "synth256", "random:<seed>:<n>" (scenes/scene_builders.inc).
 * Returns 0, or TCRT_ERR_INVALID for an unknown name. */
int tcrt_hscene_build(tcrt_hscene* s, tcrt_hcamera* c, const char* name);

/* Primitives; each returns the new object's index, or TCRT_ERR_INVALID when the scene is
 * full (Scene::addObject refuses at MAX_OBJECT_COUNT-1 = 3999 objects). */
int tcrt_hscene_add_sphere(tcrt_hscene* s, const float* origin3, float radius);              /* SceneSphere(o, r) */
int tcrt_hscene_add_infinite_plane(tcrt_hscene* s, const float* origin3, const float* normal3,
                                   const float* horizontal3);                                 /* SceneInfinitePlane(o,n,h) */
int tcrt_hscene_add_finite_plane_corners(tcrt_hscene* s, const float* origin3, const float* vertical_corner3,
                                         const float* horizontal_corner3);                    /* SceneFinitePlane(o,vc,hc) */
int tcrt_hscene_add_finite_plane_axes(tcrt_hscene* s, const float* origin3, const float* normal3,
                                      const float* horizontal3, float v_dist, float h_dist);  /* SceneFinitePlane(o,n,h,v,h) */
/* Scene::makeSceneBox + addObject of its 6 faces; returns index of the first face */
int tcrt_hscene_add_box(tcrt_hscene* s, const float* origin3, const float* dims3);
int tcrt_hscene_object_count(const tcrt_hscene* s);                                          /* Scene::getObjectCount */

/* Per-object setters (obj = index returned above); 0 or TCRT_ERR_INVALID */
int tcrt_hobj_set_color(tcrt_hscene* s, int obj, float r, float g, float b);                 /* ObjMaterial::setColor */
int tcrt_hobj_set_diffuse(tcrt_hscene* s, int obj, float f);                                 /* setDiffuseFactor */
int tcrt_hobj_set_specular(tcrt_hscene* s, int obj, float f);                                /* setSpecularFactor */
int tcrt_hobj_set_reflective(tcrt_hscene* s, int obj, float f);                              /* setReflectiveFactor */
int tcrt_hobj_set_light(tcrt_hscene* s, int obj, float intensity);                           /* setAsLightSource + setIntensity */
int tcrt_hobj_set_checker(tcrt_hscene* s, int obj, const float* light_rgb3, const float* dark_rgb3, float width,
                          float height);                                                     /* Texture_CheckerBoard + setTexture */

/* Text scene description -> the same construction calls (SURVEY §8f: the reference hard-codes its
 * scenes and lists a loader as a TODO, rt_project_parameters.h:31-32).  One statement per line,
 * '#' starts a comment, numbers are C floats (decimal or hex-float):
 *   sphere cx cy cz r | infinite_plane o(3) n(3) h(3) | finite_plane_corners o(3) vcorner(3) hcorner(3)
 *   finite_plane_axes o(3) n(3) h(3) v_dist h_dist | box o(3) dims(3)          -- primitives
 *   color r g b | diffuse f | specular f | reflective f | light intensity
 *   checker lr lg lb dr dg db width height            -- apply to the objects of the last primitive line
 *   camera two_mirrors                                -- Camera::setSceneTwoMirrors()
 * Returns 0, or TCRT_ERR_INVALID / TCRT_ERR_IO with a message ("line N: ...") in err (may be NULL). */
int tcrt_hscene_load_text(tcrt_hscene* s, tcrt_hcamera* c, const char* path, char* err, size_t err_cap);

/* Scene::flatten(): fills *out with pointers into storage owned by the handle, valid until
 * the next flatten / mutation / free of the handle. */
int tcrt_hscene_flatten(tcrt_hscene* s, tcrt_scene* out);

#ifdef __cplusplus
}
#endif
#endif /* TCRT_HOST_H_ */
