// include/CelioRayTracer.hpp — host-side construction API of the B200 render path.
//
// Same namespace, class names, constructor signatures and setter/getter names as the
// reference's public surface (SURVEY.md §8b), so scene-building code written for
// ccelio/TileCodeRayTracer compiles unchanged (scenes/scene_builders.inc is compiled
// against both).  What is different by design:
//   * objects are plain data; there is no virtual collision() (SceneObject.h:166) and no
//     CollisionObject — intersection, shading and recursion run on the GPU behind
//     include/tcrt.h.  Each primitive instead knows how to append itself to the per-type
//     structure-of-arrays (SceneFlattener) that tcrt_upload_scene consumes.
//   * everything the reference derives in its constructors (normalised axes, r*r,
//     -(origin.normal), reverse normals, moved light origin) is derived here with the same
//     float operations in the same order, on the host, once.  This TU must be compiled
//     with FP contraction off (-ffp-contract=off): the values are part of the parity
//     contract.
// Reference locations are cited per class.
#ifndef CELIO_RAYTRACER_HPP_
#define CELIO_RAYTRACER_HPP_

#include <math.h>
#include <stdio.h>
#include <vector>

#include "tcrt.h"

namespace CelioRayTracer {

typedef float sdecimal32;  // rt_project_parameters.h:41 (USING_FIXED_POINT false)

// ---- vector3d.h:31-124 ---------------------------------------------------------------
// Three binary32 members; every operator is the obvious per-component float operation
// with no reassociation.  normalize() is one sqrtf and three IEEE divisions
// (vector3d.h:57-74), not a reciprocal multiply.
class vector3d {
public:
    union {
        struct { float x, y, z; };
        struct { float r, g, b; };
        struct { float red, grn, blue; };
    };
    vector3d() { x = 0.0f; y = 0.0f; z = 0.0f; }
    vector3d(sdecimal32 ax, sdecimal32 ay, sdecimal32 az) { x = ax; y = ay; z = az; }

    void normalize() {
        const float len = sqrtf(x * x + y * y + z * z);
        x = x / len;
        y = y / len;
        z = z / len;
    }
    float length() const { return sqrtf(x * x + y * y + z * z); }
    float dot(const vector3d& v) const { return x * v.x + y * v.y + z * v.z; }
    // this = a x b   (vector3d.h:101-104)
    void cross(const vector3d& a, const vector3d& b) {
        const float cx = a.y * b.z - a.z * b.y;
        const float cy = a.z * b.x - a.x * b.z;
        const float cz = a.x * b.y - a.y * b.x;
        x = cx; y = cy; z = cz;
    }
    void operator+=(const vector3d& v) { x += v.x; y += v.y; z += v.z; }
    void operator-=(const vector3d& v) { x -= v.x; y -= v.y; z -= v.z; }
    void operator*=(float f) { x *= f; y *= f; z *= f; }
    // the reference negates as 0 - c (vector3d.h:113): +0 stays +0
    vector3d operator-() const { return vector3d(0.0f - x, 0.0f - y, 0.0f - z); }
};
inline vector3d operator+(const vector3d& a, const vector3d& b) { return vector3d(a.x + b.x, a.y + b.y, a.z + b.z); }
inline vector3d operator-(const vector3d& a, const vector3d& b) { return vector3d(a.x - b.x, a.y - b.y, a.z - b.z); }
inline vector3d operator*(const vector3d& v, sdecimal32 f) { return vector3d(v.x * f, v.y * f, v.z * f); }
inline vector3d operator*(sdecimal32 f, const vector3d& v) { return vector3d(v.x * f, v.y * f, v.z * f); }
inline vector3d operator*(const vector3d& a, const vector3d& b) { return vector3d(a.x * b.x, a.y * b.y, a.z * b.z); }

typedef vector3d Color;  // vector3d.h:163

// ---- Color_Values.h:7-17 (declared here, defined once in the library) ------------------
extern const Color COLOR_WHITE, COLOR_RED, COLOR_YELLOW, COLOR_GREEN, COLOR_CYAN, COLOR_BLUE, COLOR_BLACK,
    COLOR_DARK_GREY, COLOR_LIGHT_GREY, COLOR_BROWN;

// ---- Ray.h:12-38: origin + direction; both non-default ctors normalise -------------------
class Ray {
public:
    Ray() : origin(0.0f, 0.0f, 0.0f), direction(1.0f, 0.0f, 0.0f) {}
    Ray(vector3d o, vector3d d) : origin(o), direction(d) { direction.normalize(); }
    Ray(vector3d o, vector3d point_final, vector3d point_init) : origin(o), direction(point_final - point_init) {
        direction.normalize();
    }
    vector3d getOrigin() const { return origin; }
    vector3d getDirection() const { return direction; }

private:
    vector3d origin;
    vector3d direction;
};

// ---- ObjTexture.h:14-56 -----------------------------------------------------------------
// The lookup itself (getTexturePixel, ObjTexture.h:31) runs on the device; a texture only
// has to describe itself to the flattener.
class ObjTexture {
public:
    ObjTexture() : width(1.0f), height(1.0f) {}
    ObjTexture(sdecimal32 w, sdecimal32 h) : width(w), height(h) {}
    virtual ~ObjTexture() {}
    void setWidth(sdecimal32 w) { width = w; }
    void setHeight(sdecimal32 h) { height = h; }
    float getWidth() const { return width; }
    float getHeight() const { return height; }
    // (light rgb, width, dark rgb, height) of a 2x2-cell checker; false = not a checker
    virtual bool describeChecker(float out8[8]) const = 0;

protected:
    float width;
    float height;
};

// ---- Texture_CheckerBoard.h:13-71: default tile 2x2, white / black ---------------------------
class Texture_CheckerBoard : public ObjTexture {
public:
    Texture_CheckerBoard();
    Texture_CheckerBoard(Color l, Color d);
    void setLightColor(Color l) { light_color = l; }
    void setDarkColor(Color d) { dark_color = d; }
    bool describeChecker(float out8[8]) const;

private:
    Color light_color;
    Color dark_color;
};

// ---- ObjMaterial.h:10-82: white, diffuse 1, specular 1, reflective 0 -----------------------
class ObjMaterial {
public:
    ObjMaterial()
        : myColor(1.0f, 1.0f, 1.0f), myObjTexture_ptr(NULL), absorption_factor(0.0f), diffuse_factor(1.0f),
          specular_factor(1.0f), reflective_factor(0.0f), refractive_factor(0.0f) {}
    void setColor(vector3d c) { myColor = c; }
    void setDiffuseFactor(float d) { diffuse_factor = d; }
    void setSpecularFactor(float s) { specular_factor = s; }
    // The reference only warns when absorption+reflective+refractive > 1 (ObjMaterial.h:31-57).
    void setAbsorptionFactor(float a) { absorption_factor = a; warnIfOverUnity("Absorption"); }
    void setReflectiveFactor(float k) { reflective_factor = k; warnIfOverUnity("Reflective"); }
    void setRefractiveFactor(float k) { refractive_factor = k; warnIfOverUnity("Refractive"); }
    void setTexture(ObjTexture* t) { myObjTexture_ptr = t; }
    vector3d getColor() const { return myColor; }
    ObjTexture* getTexture() const { return myObjTexture_ptr; }
    float getDiffuseFactor() const { return diffuse_factor; }
    float getSpecularFactor() const { return specular_factor; }
    float getAbsorptionFactor() const { return absorption_factor; }
    float getReflectiveFactor() const { return reflective_factor; }
    float getRefractiveFactor() const { return refractive_factor; }

private:
    void warnIfOverUnity(const char* which) const {
        if ((absorption_factor + reflective_factor + refractive_factor) > 1)
            fprintf(stderr, "***ERROR. Setting %s Factor.\n Ab: %f\n Refl: %f\n Refr: %f\n", which, absorption_factor,
                    reflective_factor, refractive_factor);
    }
    Color myColor;
    ObjTexture* myObjTexture_ptr;
    float absorption_factor, diffuse_factor, specular_factor, reflective_factor, refractive_factor;
};

class SceneFlattener;  // below

// ---- SceneObject.h:154-203, SceneObject.cpp:9-27 ---------------------------------------------
class SceneObject {
public:
    SceneObject();                       // diffuse 0.25 (SceneObject.cpp:16)
    explicit SceneObject(vector3d o);    // material defaults (diffuse 1)
    virtual ~SceneObject() {}

    ObjMaterial* getMaterial() { return &myMaterial; }
    void moveOrigin(sdecimal32 dx, sdecimal32 dy, sdecimal32 dz) { origin.x += dx; origin.y += dy; origin.z += dz; }
    void changeOrigin(vector3d o) { origin = o; }
    vector3d getOrigin() const { return origin; }
    void setIndex(int i) { my_object_index = i; }
    int getIndex() const { return my_object_index; }
    void setAsLightSource() { isaLightSource = true; }
    bool checkIsaLightSource() const { return isaLightSource; }
    void setIntensity(sdecimal32 d) { intensity = d; }
    sdecimal32 getIntensity() const { return intensity; }

    // Replaces virtual collision(Ray*): append this primitive's test data to its type's SoA.
    virtual void flattenGeometry(SceneFlattener& out, int object_index) const = 0;

protected:
    ObjMaterial myMaterial;
    vector3d origin;
    bool isaLightSource;
    sdecimal32 intensity;
    int my_object_index;
};

// ---- SceneSphere.h / SceneSphere.cpp:38-48 ---------------------------------------------------
class SceneSphere : public SceneObject {
public:
    SceneSphere();
    SceneSphere(vector3d _origin, sdecimal32 _radius);
    void flattenGeometry(SceneFlattener& out, int object_index) const;

private:
    sdecimal32 radius;
    sdecimal32 radius_squared;
};

// ---- SceneInfinitePlane.h / SceneInfinitePlane.cpp:7-26 ----------------------------------------
class SceneInfinitePlane : public SceneObject {
public:
    SceneInfinitePlane();
    SceneInfinitePlane(vector3d o, vector3d n, vector3d h);
    void flattenGeometry(SceneFlattener& out, int object_index) const;

private:
    vector3d normal, vertical, horizontal, reverseNormal;
    sdecimal32 distance_to_origin;
};

// ---- SceneFinitePlane.h / SceneFinitePlane.cpp:13-80 --------------------------------------------
class SceneFinitePlane : public SceneObject {
public:
    SceneFinitePlane();
    // three corners; origin must be the corner between the other two (SceneFinitePlane.cpp:49-80)
    SceneFinitePlane(vector3d _origin, vector3d _vertical_corner, vector3d _horizontal_corner);
    // (origin, normal, horizontal axis, vertical extent, horizontal extent) — the meaning the
    // reference's definition gives the arguments (SceneFinitePlane.cpp:18-19)
    SceneFinitePlane(vector3d _origin, vector3d _normal, vector3d _horizontal, float v_dist, float h_dist);
    void flattenGeometry(SceneFlattener& out, int object_index) const;

private:
    vector3d plane_origin, normal, vertical, horizontal, reverseNormal;
    sdecimal32 v_distance, h_distance, distance_to_origin;
};

// ---- Camera.h / Camera.cpp -------------------------------------------------------------------------
class Camera {
public:
    Camera();                                   // fixed pose, Camera.cpp:9-40
    Ray* createEyeRay(sdecimal32 dx_percent, sdecimal32 dy_percent) const;  // Camera.cpp:71-84 (caller frees)
    sdecimal32 getScreenWidth() const { return screen_width; }
    sdecimal32 getScreeHeight() const { return screen_height; }
    void setSceneTwoMirrors();                  // Camera.cpp:42-69
    // the pose arithmetic of Camera.cpp:22-38: screen centre so, screen x axis horiz, view direction outward (neither
    // normalised); vertical = horiz x outward, all three normalised, the eye one unit behind the screen.  The screen size
    // is kept (another field of view: edit the exported tcrt_camera's screen_* fields, halfwidth = width / 2).
    void aim(vector3d so, vector3d horiz, vector3d outward);
    // what the kernels read for primary-ray generation
    void exportTo(tcrt_camera* out) const;

private:
    sdecimal32 screen_width, screen_height, screen_halfwidth, screen_halfheight;
    vector3d screen_origin, vector_outwards, vector_vertical, vector_horizontal;
    sdecimal32 eye_distance;
    vector3d eye_origin;
};

// ---- flattened scene (owner of the arrays a tcrt_scene points into) -----------------------------------
class SceneFlattener {
public:
    std::vector<float> sphere_geom, fin_geom, inf_geom;
    std::vector<int> sphere_obj, fin_obj, inf_obj;
    std::vector<float> obj_surface, obj_material, obj_origin, obj_normals, textures;
    std::vector<int> obj_info, light_obj;
    int n_objects;
    SceneFlattener() : n_objects(0) {}
    // called by flattenGeometry(); return the slot within the type
    int addSphere(int obj, vector3d c, float r2);
    int addFinitePlane(int obj, vector3d n, float neg_dto, vector3d h, float h_dist, vector3d v, float v_dist,
                       vector3d plane_origin, vector3d reverse_n);
    int addInfinitePlane(int obj, vector3d n, float neg_dto, vector3d h, vector3d v, vector3d origin,
                         vector3d reverse_n);
    tcrt_scene view() const;  // valid while *this is alive and unmodified
private:
    void setInfo(int obj, int type, int slot, vector3d n, vector3d rn);
};

// ---- Scene.h / Scene.cpp ------------------------------------------------------------------------------
#define MAX_OBJECT_COUNT 4000  // Scene.h:8
class Scene {
public:
    Scene();
    virtual ~Scene();
    int initialize(void);                       // the default "museum", Scene.cpp:209-387
    int initializeTwoMirrors(Camera* myCamera); // Scene.cpp:23-206
    int getObjectCount() const { return object_count; }
    void addObject(SceneObject* new_obj_ptr);   // refuses at MAX_OBJECT_COUNT-1 with a message, Scene.cpp:470-479
    SceneObject* getObject(int i) const { return objects[i]; }
    SceneFinitePlane** makeSceneBox(vector3d _origin, vector3d _dims);  // Scene.cpp:392-416
    // New: the per-type SoA export consumed by tcrt_upload_scene.
    void flatten(SceneFlattener& out) const;

private:
    SceneObject** objects;
    int object_count;
};

}  // namespace CelioRayTracer

#endif  // CELIO_RAYTRACER_HPP_
