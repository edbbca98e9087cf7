// tcrt_cluster.cpp — host side of the box-cluster culling structure for axis-aligned finite planes.
//
// Scene::makeSceneBox (Scene.cpp:392-416) builds every box of the reference's scenes out of six
// SceneFinitePlane objects whose normal / horizontal / vertical vectors are +-unit axes after the
// constructor's normalisation (SceneFinitePlane.cpp:49-80).  For such a plane the reference's test
// (SceneFinitePlane.cpp:86-123) accepts the points of an axis-aligned rectangle: coordinate i fixed
// at c = s*(-dto) (s = sign of the normal), the other two inside [origin, origin +- extent].
//
// The kernel exploits this only to PRUNE: rectangles are grouped into boxes ("clusters", at most two
// rectangles per axis) whose hull is tight for every member; a ray is slab-tested against the hull
// (inflated per ray, see tcrt_render.cu `clu_ray`) and a member becomes a candidate only if its
// plane is crossed inside the hull's cross-section.  Candidates are then evaluated with the
// reference's exact arithmetic from the ordinary finite-plane record, so results cannot change.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "tcrt_device.h"

namespace {

struct ARect {
    int plane;        // index into the caller's plane list
    int axis;         // normal axis
    float c;          // plane coordinate on that axis, exactly s * (-dto)
    double lo[3], hi[3];   // accepted region (lo[axis] == hi[axis] == c)
};

// +-unit axis vector: exactly one component of magnitude 1, the others (signed) zero
bool unit_axis(const float* v, int& axis, float& sign) {
    int a = -1;
    for (int k = 0; k < 3; k++) {
        if (v[k] == 0.0f) continue;
        if (a >= 0 || (v[k] != 1.0f && v[k] != -1.0f)) return false;
        a = k;
    }
    if (a < 0) return false;
    axis = a;
    sign = v[a];
    return true;
}

bool classify(const float* g, int plane, ARect& r) {
    for (int k = 0; k < 16; k++)
        if (k != 15 && !std::isfinite(g[k])) return false;
    int an, ah, av;
    float sn, sh, sv;
    if (!unit_axis(g, an, sn) || !unit_axis(g + 4, ah, sh) || !unit_axis(g + 8, av, sv)) return false;
    if (an == ah || an == av || ah == av) return false;
    const float hd = g[7], vd = g[11];
    if (!(hd >= 0.0f) || !(vd >= 0.0f)) return false;
    r.plane = plane;
    r.axis = an;
    r.c = sn * g[3];   // exact: multiplication by +-1
    r.lo[an] = r.hi[an] = (double)r.c;
    // 0 <= sh*(P - po)[ah] <= hd   (SceneFinitePlane.cpp:116-122 with h = sh * e_ah)
    r.lo[ah] = (double)g[12 + ah] + (sh > 0 ? 0.0 : -(double)hd);
    r.hi[ah] = (double)g[12 + ah] + (sh > 0 ? (double)hd : 0.0);
    r.lo[av] = (double)g[12 + av] + (sv > 0 ? 0.0 : -(double)vd);
    r.hi[av] = (double)g[12 + av] + (sv > 0 ? (double)vd : 0.0);
    return true;
}

struct Cluster {
    double lo[3], hi[3];
    std::vector<int> members;   // indices into the ARect list
    int per_axis[3] = {0, 0, 0};
};

float round_down(double d) {
    float f = (float)d;
    if ((double)f > d) f = nextafterf(f, -INFINITY);
    return f;
}
float round_up(double d) {
    float f = (float)d;
    if ((double)f < d) f = nextafterf(f, INFINITY);
    return f;
}

}  // namespace

void tcrt_build_box_clusters(const float* fin_geom, const std::vector<int>& planes, std::vector<int>& arect_of_plane,
                             std::vector<TcrtBoxCluster>& out) {
    out.clear();
    arect_of_plane.assign(planes.size(), 0);
    std::vector<ARect> rects;
    double scale = 1.0;
    for (size_t p = 0; p < planes.size(); p++) {
        ARect r;
        if (!classify(fin_geom + 16 * (size_t)planes[p], (int)p, r)) continue;
        rects.push_back(r);
        arect_of_plane[p] = 1;
        for (int k = 0; k < 3; k++) scale = std::max(scale, std::max(fabs(r.lo[k]), fabs(r.hi[k])));
    }
    const double tol = 1e-4 * scale;
    // greedy: a rectangle joins the first cluster whose hull stays tight for every member
    std::vector<Cluster> clusters;
    auto tight = [&](const Cluster& c, const double* lo, const double* hi) {
        for (int m : c.members) {
            const ARect& r = rects[m];
            for (int k = 0; k < 3; k++) {
                if (k == r.axis) continue;
                if (fabs(r.lo[k] - lo[k]) > tol || fabs(r.hi[k] - hi[k]) > tol) return false;
            }
        }
        return true;
    };
    for (size_t i = 0; i < rects.size(); i++) {
        const ARect& r = rects[i];
        bool placed = false;
        for (auto& c : clusters) {
            if (c.per_axis[r.axis] >= 2) continue;
            double lo[3], hi[3];
            for (int k = 0; k < 3; k++) {
                lo[k] = std::min(c.lo[k], r.lo[k]);
                hi[k] = std::max(c.hi[k], r.hi[k]);
            }
            c.members.push_back((int)i);
            const bool ok = tight(c, lo, hi);
            if (!ok) {
                c.members.pop_back();
                continue;
            }
            memcpy(c.lo, lo, sizeof lo);
            memcpy(c.hi, hi, sizeof hi);
            c.per_axis[r.axis]++;
            placed = true;
            break;
        }
        if (!placed) {
            Cluster c;
            memcpy(c.lo, r.lo, sizeof c.lo);
            memcpy(c.hi, r.hi, sizeof c.hi);
            c.members.push_back((int)i);
            c.per_axis[r.axis] = 1;
            clusters.push_back(c);
        }
    }
    // small boxes first: objects inside a room are nearer than its walls, so `best` shrinks early
    auto measure = [](const Cluster& c) {
        double dx = c.hi[0] - c.lo[0], dy = c.hi[1] - c.lo[1], dz = c.hi[2] - c.lo[2];
        return dx * dy + dy * dz + dz * dx;
    };
    std::stable_sort(clusters.begin(), clusters.end(),
                     [&](const Cluster& a, const Cluster& b) { return measure(a) < measure(b); });
    for (const Cluster& c : clusters) {
        TcrtBoxCluster o;
        for (int k = 0; k < 3; k++) {
            o.lo[k] = round_down(c.lo[k]);
            o.hi[k] = round_up(c.hi[k]);
        }
        for (int f = 0; f < 6; f++) {
            o.c[f] = NAN;      // absent face: every comparison with it is false
            o.plane[f] = -1;
        }
        int used[3] = {0, 0, 0};
        for (int m : c.members) {
            const ARect& r = rects[m];
            const int f = 2 * r.axis + used[r.axis]++;
            o.c[f] = r.c;
            o.plane[f] = r.plane;
        }
        out.push_back(o);
    }
}

bool tcrt_refit_box_cluster(const float* fin_slots, TcrtBoxCluster& c) {
    // the builder's hull of the members' rectangles (contained, not necessarily tight: DESIGN.md §4.5 "Moving planes")
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    float face[6];
    for (int f = 0; f < 6; f++) {
        face[f] = NAN;
        if (c.plane[f] < 0) continue;
        ARect r;
        if (!classify(fin_slots + 16 * (size_t)c.plane[f], c.plane[f], r) || r.axis != f / 2) return false;
        for (int k = 0; k < 3; k++) {
            lo[k] = std::min(lo[k], r.lo[k]);
            hi[k] = std::max(hi[k], r.hi[k]);
        }
        face[f] = r.c;
    }
    for (int k = 0; k < 3; k++) {
        c.lo[k] = round_down(lo[k]);
        c.hi[k] = round_up(hi[k]);
    }
    memcpy(c.c, face, sizeof face);
    return true;
}
