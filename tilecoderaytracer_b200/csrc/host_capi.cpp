// host_capi.cpp — include/tcrt_host.h: C binding of the host construction API.
#include "tcrt_host.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "CelioRayTracer.hpp"
#include "scene_builders.inc"

using namespace CelioRayTracer;

struct tcrt_hscene {
    Scene scene;
    SceneFlattener flat;
};
struct tcrt_hcamera {
    Camera cam;
};

static vector3d v3(const float* p) { return vector3d(p[0], p[1], p[2]); }

extern "C" {

tcrt_hscene* tcrt_hscene_new(void) { return new tcrt_hscene(); }
void tcrt_hscene_free(tcrt_hscene* s) {
    if (!s) return;
    // the handle owns the objects it was given (the reference never frees them)
    for (int i = 0; i < s->scene.getObjectCount(); i++) delete s->scene.getObject(i);
    delete s;
}
tcrt_hcamera* tcrt_hcamera_new(void) { return new tcrt_hcamera(); }
void tcrt_hcamera_free(tcrt_hcamera* c) { delete c; }
void tcrt_hcamera_set_two_mirrors(tcrt_hcamera* c) { if (c) c->cam.setSceneTwoMirrors(); }
void tcrt_hcamera_aim(tcrt_hcamera* c, const float* so, const float* h, const float* o) {
    if (c && so && h && o) c->cam.aim(v3(so), v3(h), v3(o));
}
void tcrt_hcamera_export(const tcrt_hcamera* c, tcrt_camera* out) { if (c && out) c->cam.exportTo(out); }
void tcrt_hcamera_eye_ray(const tcrt_hcamera* c, float dx, float dy, float* o3, float* d3) {
    Ray* r = c->cam.createEyeRay(dx, dy);
    vector3d o = r->getOrigin(), d = r->getDirection();
    delete r;
    o3[0] = o.x; o3[1] = o.y; o3[2] = o.z;
    d3[0] = d.x; d3[1] = d.y; d3[2] = d.z;
}

int tcrt_hscene_build(tcrt_hscene* s, tcrt_hcamera* c, const char* name) {
    if (!s || !name) return TCRT_ERR_INVALID;
    if (!strcmp(name, "default")) return s->scene.initialize() ? TCRT_ERR_INVALID : TCRT_OK;
    if (!strcmp(name, "two_mirrors")) {
        if (!c) return TCRT_ERR_INVALID;
        return s->scene.initializeTwoMirrors(&c->cam) ? TCRT_ERR_INVALID : TCRT_OK;
    }
    if (!strcmp(name, "synth1024")) { tcrt_scenes::build_synth1024(s->scene); return TCRT_OK; }
    if (!strcmp(name, "synth256")) { tcrt_scenes::build_synth256(s->scene); return TCRT_OK; }
    if (!strncmp(name, "random:", 7)) {
        unsigned int seed = 0;
        int n = 0;
        if (sscanf(name + 7, "%u:%d", &seed, &n) != 2 || n < 1) return TCRT_ERR_INVALID;
        tcrt_scenes::build_random(s->scene, seed, n);
        return TCRT_OK;
    }
    if (!strncmp(name, "lattice:", 8)) {
        unsigned int seed = 0;
        int n = 0;
        if (sscanf(name + 8, "%u:%d", &seed, &n) != 2 || n < 1 || n > 30) return TCRT_ERR_INVALID;
        tcrt_scenes::build_lattice(s->scene, seed, n);
        return TCRT_OK;
    }
    if (!strncmp(name, "boxes:", 6)) {
        unsigned int seed = 0;
        int n = 0;
        if (sscanf(name + 6, "%u:%d", &seed, &n) != 2 || n < 0) return TCRT_ERR_INVALID;
        tcrt_scenes::build_boxes(s->scene, seed, n);
        return TCRT_OK;
    }
    return TCRT_ERR_INVALID;
}

static int add(tcrt_hscene* s, SceneObject* o) {
    int before = s->scene.getObjectCount();
    o->setIndex(before);
    s->scene.addObject(o);
    if (s->scene.getObjectCount() == before) { delete o; return TCRT_ERR_INVALID; }
    return before;
}
int tcrt_hscene_add_sphere(tcrt_hscene* s, const float* o, float radius) {
    if (!s || !o) return TCRT_ERR_INVALID;
    return add(s, new SceneSphere(v3(o), radius));
}
int tcrt_hscene_add_infinite_plane(tcrt_hscene* s, const float* o, const float* n, const float* h) {
    if (!s || !o || !n || !h) return TCRT_ERR_INVALID;
    return add(s, new SceneInfinitePlane(v3(o), v3(n), v3(h)));
}
int tcrt_hscene_add_finite_plane_corners(tcrt_hscene* s, const float* o, const float* vc, const float* hc) {
    if (!s || !o || !vc || !hc) return TCRT_ERR_INVALID;
    return add(s, new SceneFinitePlane(v3(o), v3(vc), v3(hc)));
}
int tcrt_hscene_add_finite_plane_axes(tcrt_hscene* s, const float* o, const float* n, const float* h, float v_dist,
                                      float h_dist) {
    if (!s || !o || !n || !h) return TCRT_ERR_INVALID;
    return add(s, new SceneFinitePlane(v3(o), v3(n), v3(h), v_dist, h_dist));
}
int tcrt_hscene_add_box(tcrt_hscene* s, const float* o, const float* d) {
    if (!s || !o || !d) return TCRT_ERR_INVALID;
    if (s->scene.getObjectCount() + 7 >= MAX_OBJECT_COUNT) return TCRT_ERR_INVALID;
    SceneFinitePlane** faces = s->scene.makeSceneBox(v3(o), v3(d));
    int first = s->scene.getObjectCount();
    for (int f = 0; f < 6; f++) add(s, faces[f]);
    delete[] faces;
    return first;
}
int tcrt_hscene_object_count(const tcrt_hscene* s) { return s ? s->scene.getObjectCount() : TCRT_ERR_INVALID; }

static SceneObject* obj_at(tcrt_hscene* s, int i) {
    if (!s || i < 0 || i >= s->scene.getObjectCount()) return NULL;
    return s->scene.getObject(i);
}
int tcrt_hobj_set_color(tcrt_hscene* s, int i, float r, float g, float b) {
    SceneObject* o = obj_at(s, i);
    if (!o) return TCRT_ERR_INVALID;
    o->getMaterial()->setColor(Color(r, g, b));
    return TCRT_OK;
}
int tcrt_hobj_set_diffuse(tcrt_hscene* s, int i, float f) {
    SceneObject* o = obj_at(s, i);
    if (!o) return TCRT_ERR_INVALID;
    o->getMaterial()->setDiffuseFactor(f);
    return TCRT_OK;
}
int tcrt_hobj_set_specular(tcrt_hscene* s, int i, float f) {
    SceneObject* o = obj_at(s, i);
    if (!o) return TCRT_ERR_INVALID;
    o->getMaterial()->setSpecularFactor(f);
    return TCRT_OK;
}
int tcrt_hobj_set_reflective(tcrt_hscene* s, int i, float f) {
    SceneObject* o = obj_at(s, i);
    if (!o) return TCRT_ERR_INVALID;
    o->getMaterial()->setReflectiveFactor(f);
    return TCRT_OK;
}
int tcrt_hobj_set_light(tcrt_hscene* s, int i, float intensity) {
    SceneObject* o = obj_at(s, i);
    if (!o) return TCRT_ERR_INVALID;
    o->setAsLightSource();
    o->setIntensity(intensity);
    return TCRT_OK;
}
int tcrt_hobj_set_checker(tcrt_hscene* s, int i, const float* l, const float* d, float width, float height) {
    SceneObject* o = obj_at(s, i);
    if (!o || !l || !d) return TCRT_ERR_INVALID;
    ObjTexture* t = new Texture_CheckerBoard(Color(l[0], l[1], l[2]), Color(d[0], d[1], d[2]));
    t->setHeight(height);
    t->setWidth(width);
    o->getMaterial()->setTexture(t);   // like the reference, textures are never freed
    return TCRT_OK;
}

int tcrt_hscene_load_text(tcrt_hscene* s, tcrt_hcamera* c, const char* path, char* err, size_t err_cap) {
    auto fail = [&](int code, int line, const char* msg) {
        if (err && err_cap) snprintf(err, err_cap, "line %d: %s", line, msg);
        return code;
    };
    if (!s || !path) return fail(TCRT_ERR_INVALID, 0, "null argument");
    FILE* f = fopen(path, "r");
    if (!f) return fail(TCRT_ERR_IO, 0, "cannot open scene file");
    char buf[1024];
    int line = 0, first = -1, count = 0;   // objects created by the last primitive line
    int rc = TCRT_OK;
    while (rc == TCRT_OK && fgets(buf, sizeof buf, f)) {
        line++;
        if (char* hash = strchr(buf, '#')) *hash = 0;
        char* save = NULL;
        char* kw = strtok_r(buf, " \t\r\n", &save);
        if (!kw) continue;
        float v[16];
        int n = 0;
        char* tok;
        bool bad = false;
        char word[64] = "";
        while ((tok = strtok_r(NULL, " \t\r\n", &save)) != NULL) {
            char* end = NULL;
            float x = strtof(tok, &end);
            if (end == tok || *end != 0) {
                if (n == 0 && !word[0]) { snprintf(word, sizeof word, "%s", tok); continue; }
                bad = true;
                break;
            }
            if (n < 16) v[n] = x;
            n++;
        }
        if (bad) { rc = fail(TCRT_ERR_INVALID, line, "not a number"); break; }
        auto need = [&](int k) { return n == k && !word[0]; };
        auto created = [&](int idx, int cnt) {
            if (idx < 0) return fail(TCRT_ERR_INVALID, line, "scene is full");
            first = idx;
            count = cnt;
            return (int)TCRT_OK;
        };
        auto each = [&](int (*fn)(tcrt_hscene*, int, float), float x) {
            if (first < 0) return fail(TCRT_ERR_INVALID, line, "material statement before any primitive");
            for (int i = first; i < first + count; i++) fn(s, i, x);
            return (int)TCRT_OK;
        };
        if (!strcmp(kw, "sphere") && need(4)) rc = created(tcrt_hscene_add_sphere(s, v, v[3]), 1);
        else if (!strcmp(kw, "infinite_plane") && need(9)) rc = created(tcrt_hscene_add_infinite_plane(s, v, v + 3, v + 6), 1);
        else if (!strcmp(kw, "finite_plane_corners") && need(9))
            rc = created(tcrt_hscene_add_finite_plane_corners(s, v, v + 3, v + 6), 1);
        else if (!strcmp(kw, "finite_plane_axes") && need(11))
            rc = created(tcrt_hscene_add_finite_plane_axes(s, v, v + 3, v + 6, v[9], v[10]), 1);
        else if (!strcmp(kw, "box") && need(6)) rc = created(tcrt_hscene_add_box(s, v, v + 3), 6);
        else if (!strcmp(kw, "diffuse") && need(1)) rc = each(tcrt_hobj_set_diffuse, v[0]);
        else if (!strcmp(kw, "specular") && need(1)) rc = each(tcrt_hobj_set_specular, v[0]);
        else if (!strcmp(kw, "reflective") && need(1)) rc = each(tcrt_hobj_set_reflective, v[0]);
        else if (!strcmp(kw, "light") && need(1)) rc = each(tcrt_hobj_set_light, v[0]);
        else if (!strcmp(kw, "color") && need(3)) {
            if (first < 0) rc = fail(TCRT_ERR_INVALID, line, "material statement before any primitive");
            for (int i = first; rc == TCRT_OK && i < first + count; i++) tcrt_hobj_set_color(s, i, v[0], v[1], v[2]);
        } else if (!strcmp(kw, "checker") && need(8)) {
            if (first < 0) rc = fail(TCRT_ERR_INVALID, line, "material statement before any primitive");
            for (int i = first; rc == TCRT_OK && i < first + count; i++) tcrt_hobj_set_checker(s, i, v, v + 3, v[6], v[7]);
        } else if (!strcmp(kw, "camera") && n == 0 && !strcmp(word, "two_mirrors")) {
            if (!c) rc = fail(TCRT_ERR_INVALID, line, "no camera handle given");
            else tcrt_hcamera_set_two_mirrors(c);
        } else {
            rc = fail(TCRT_ERR_INVALID, line, "unknown statement or wrong number of arguments");
        }
    }
    fclose(f);
    return rc;
}

int tcrt_hscene_flatten(tcrt_hscene* s, tcrt_scene* out) {
    if (!s || !out) return TCRT_ERR_INVALID;
    s->scene.flatten(s->flat);
    *out = s->flat.view();
    return TCRT_OK;
}

}  // extern "C"
