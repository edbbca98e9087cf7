// tcrt_bvh.cpp — host-side BVH builder for the render kernel's culling structure.
//
// The reference tests every object for every ray (getCollision, RayTracer.cpp:73-86); its author
// lists "octree parsing" as not supported (README.md:25-29).  The BVH here is only a pruning
// device: the kernel still evaluates the reference's exact arithmetic for every primitive whose
// (inflated) box the ray may touch, so results are unchanged (see tcrt_render.cu).
//
// Binary tree, surface-area heuristic with a full sweep on each axis, leaves of <= 4 primitives
// (<= 8 when splitting does not pay), depth capped at 40 by falling back to median splits.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "tcrt_device.h"

namespace {

struct Box {
    float lo[3], hi[3];
    void reset() {
        for (int k = 0; k < 3; k++) { lo[k] = INFINITY; hi[k] = -INFINITY; }
    }
    void grow(const float* b) {
        for (int k = 0; k < 3; k++) {
            lo[k] = std::min(lo[k], b[k]);
            hi[k] = std::max(hi[k], b[3 + k]);
        }
    }
    double area() const {
        double dx = (double)hi[0] - lo[0], dy = (double)hi[1] - lo[1], dz = (double)hi[2] - lo[2];
        if (!(dx >= 0) || !(dy >= 0) || !(dz >= 0)) return 0.0;
        if (!std::isfinite(dx) || !std::isfinite(dy) || !std::isfinite(dz)) return 1e300;
        return 2.0 * (dx * dy + dy * dz + dz * dx);
    }
};

struct Builder {
    const float* boxes;            // n x 6
    std::vector<int>& order;       // permuted in place
    std::vector<float4>& nodes;
    std::vector<double> suffix;
    int max_depth = 0;
    int max_leaf = 4;   // 4 and 6 measure the same, 1-3 slower (profiles/README.md)

    Builder(const float* b, std::vector<int>& o, std::vector<float4>& n) : boxes(b), order(o), nodes(n) {}

    float centroid(int id, int axis) const {
        float lo = boxes[6 * id + axis], hi = boxes[6 * id + 3 + axis];
        if (!std::isfinite(lo) || !std::isfinite(hi)) return 0.f;
        return 0.5f * (lo + hi);
    }
    Box bounds(int first, int count) const {
        Box b;
        b.reset();
        for (int i = first; i < first + count; i++) b.grow(boxes + 6 * order[i]);
        return b;
    }
    static int leaf_ref(int first, int count) { return ~(first | (count << 24)); }

    // returns the encoded reference of the subtree over order[first, first+count)
    int build(int first, int count, int depth) {
        max_depth = std::max(max_depth, depth);
        if (count <= max_leaf) return leaf_ref(first, count);
        const Box parent = bounds(first, count);
        int best_axis = -1, best_split = -1;
        double best_cost = 1e308;
        if (depth < 32) {
            for (int axis = 0; axis < 3; axis++) {
                std::sort(order.begin() + first, order.begin() + first + count,
                          [&](int a, int b) { return centroid(a, axis) < centroid(b, axis); });
                suffix.assign(count + 1, 0.0);
                Box r;
                r.reset();
                for (int i = count - 1; i >= 1; i--) {
                    r.grow(boxes + 6 * order[first + i]);
                    suffix[i] = r.area();
                }
                Box l;
                l.reset();
                for (int i = 1; i < count; i++) {
                    l.grow(boxes + 6 * order[first + i - 1]);
                    double cost = l.area() * i + suffix[i] * (count - i);
                    if (cost < best_cost) { best_cost = cost; best_axis = axis; best_split = i; }
                }
            }
            // no split beats a leaf: keep small groups together
            if (count <= 2 * max_leaf && best_cost >= parent.area() * count) return leaf_ref(first, count);
        }
        if (best_axis < 0) {   // depth guard: balanced median split on the widest centroid axis
            float clo[3] = {INFINITY, INFINITY, INFINITY}, chi[3] = {-INFINITY, -INFINITY, -INFINITY};
            for (int i = first; i < first + count; i++)
                for (int k = 0; k < 3; k++) {
                    float c = centroid(order[i], k);
                    clo[k] = std::min(clo[k], c);
                    chi[k] = std::max(chi[k], c);
                }
            best_axis = 0;
            for (int k = 1; k < 3; k++)
                if (chi[k] - clo[k] > chi[best_axis] - clo[best_axis]) best_axis = k;
            best_split = count / 2;
        }
        const int axis = best_axis;
        std::sort(order.begin() + first, order.begin() + first + count,
                  [&](int a, int b) { return centroid(a, axis) < centroid(b, axis); });
        const int me = (int)(nodes.size() / 4);
        nodes.resize(nodes.size() + 4);
        const int c0 = build(first, best_split, depth + 1);
        const int c1 = build(first + best_split, count - best_split, depth + 1);
        const Box b0 = bounds(first, best_split), b1 = bounds(first + best_split, count - best_split);
        float4 q3;
        memcpy(&q3.x, &c0, 4);
        memcpy(&q3.y, &c1, 4);
        q3.z = q3.w = 0.f;
        nodes[4 * me + 0] = make_float4(b0.lo[0], b0.lo[1], b0.lo[2], b0.hi[0]);
        nodes[4 * me + 1] = make_float4(b0.hi[1], b0.hi[2], b1.lo[0], b1.lo[1]);
        nodes[4 * me + 2] = make_float4(b1.lo[2], b1.hi[0], b1.hi[1], b1.hi[2]);
        nodes[4 * me + 3] = q3;
        return me;
    }
};

}  // namespace

int tcrt_build_bvh(const std::vector<float>& boxes, int n, std::vector<int>& order, std::vector<float4>& nodes, int* depth) {
    order.resize(n);
    for (int i = 0; i < n; i++) order[i] = i;
    nodes.clear();
    Builder b(boxes.data(), order, nodes);
    const int root = b.build(0, n, 0);
    if (depth) *depth = b.max_depth;
    return root;
}

// ---- uniform grid over the BVH-covered spheres -------------------------------------------------------------------------------
// Scenes of many similar spheres (BASELINE configs 3 and 4: lattices of 1024 / 256 spheres) are walked faster with a 3D-DDA
// through a uniform grid than through a binary tree: a step costs a third of a tree node, and a ray meets a sphere after a few
// cells.  Like the BVH the grid only PRUNES: a sphere is registered in every cell its box — inflated by `reg_margin`, which
// must cover the per-ray fattening of the kernel (tcrt_render_common.cuh `fatten`) — overlaps, and spheres found in a cell are
// tested with the reference's exact arithmetic.  Rays whose fattening exceeds the margin (origins far from the scene) use the
// BVH, which therefore always exists next to the grid.
//   boxes: n x 6 floats (lo xyz, hi xyz) of the spheres in leaf order, already inflated like the BVH's.
// Returns false (no grid) when the spheres are too uneven for a grid to pay: more than 8 registrations per sphere on average,
// or a cell with more than 24 spheres.
bool tcrt_build_sphere_grid(const std::vector<float>& boxes, int n, TcrtSphereGrid& g) {
    g = TcrtSphereGrid{};
    if (n < 24) return false;
    double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
    std::vector<double> ext;
    ext.reserve(n);
    for (int i = 0; i < n; i++) {
        double e = 0;
        for (int k = 0; k < 3; k++) {
            const double a = boxes[6 * i + k], b = boxes[6 * i + 3 + k];
            if (!std::isfinite(a) || !std::isfinite(b) || !(b >= a)) return false;
            lo[k] = std::min(lo[k], a);
            hi[k] = std::max(hi[k], b);
            e = std::max(e, b - a);
        }
        ext.push_back(e);
    }
    std::sort(ext.begin(), ext.end());
    const double d_med = ext[n / 2], d_max = ext[n - 1];
    if (!(d_med > 0) || d_max > 4.0 * d_med) return false;            // one huge sphere would sit in every cell
    double vol = 1.0;
    for (int k = 0; k < 3; k++) vol *= std::max(hi[k] - lo[k], d_med);
    // Cell size and phase per axis.  Cost of a ray per unit of length: (cells entered) x (a DDA step + the spheres tested in
    // a cell) ~ (sum_k 1/c_k) x (S + T * n/V * prod_k(ov_k * c_k)), ov_k = cells a sphere overlaps along axis k.  A grid in
    // step with a lattice of spheres (cell = spacing, every sphere inside one cell) tests each sphere once; out of step it
    // registers a sphere in two cells per axis and tests eight times as many.  Coordinate descent over the axes: each takes the
    // (size, phase) minimising the model, sizes from 0.7 to 3 typical diameters, 32 phases, starting at one sphere per cell.
    const double guess = std::max(1.15 * d_med, cbrt(vol / n));
    const double margin = 0.02 * std::min(guess, 1.15 * d_med);
    const double kStep = 25.0, kTest = 30.0;        // instructions: one DDA step, one sphere test
    double cs[3] = {guess, guess, guess}, org[3], ovm[3] = {2.0, 2.0, 2.0};
    for (int k = 0; k < 3; k++) org[k] = lo[k] - 2.0 * margin;
    auto mean_overlap = [&](int k, double c, double o) {
        double ov = 0.0;
        for (int i = 0; i < n; i++)
            ov += floor(((double)boxes[6 * i + 3 + k] + margin - o) / c) - floor(((double)boxes[6 * i + k] - margin - o) / c) + 1.0;
        return ov / n;
    };
    auto model = [&](const double* c, const double* ov) {
        return (1.0 / c[0] + 1.0 / c[1] + 1.0 / c[2]) * (kStep + kTest * n / vol * (ov[0] * c[0]) * (ov[1] * c[1]) * (ov[2] * c[2]));
    };
    for (int k = 0; k < 3; k++) ovm[k] = mean_overlap(k, cs[k], org[k]);
    for (int round = 0; round < 3; round++) {
        for (int k = 0; k < 3; k++) {
            double best = model(cs, ovm), c_try[3] = {cs[0], cs[1], cs[2]}, ov_try[3] = {ovm[0], ovm[1], ovm[2]};
            // coarse: 40 sizes on a geometric scale; fine: +-4 % around the current size in 0.25 % steps (a lattice's own
            // spacing has to be met within a fraction of the gap between its spheres)
            const double c_now = cs[k];
            for (int ci = 0; ci < 40 + 33; ci++) {
                const double c = ci < 40 ? 0.7 * d_med * pow(3.0 / 0.7, ci / 39.0) : c_now * (1.0 + 0.0025 * (ci - 40 - 16));
                if ((hi[k] - lo[k] + 4.0 * margin) / c > 63.0) continue;                 // at most 64 cells per axis
                for (int ph = 0; ph < 32; ph++) {
                    const double o = lo[k] - 2.0 * margin - c * ph / 32.0;
                    c_try[k] = c;
                    ov_try[k] = mean_overlap(k, c, o);
                    const double f = model(c_try, ov_try);
                    if (f < best * (1.0 - 1e-9)) {
                        best = f;
                        cs[k] = c;
                        org[k] = o;
                        ovm[k] = ov_try[k];
                    }
                }
            }
        }
    }
    int dims[3];
    for (int k = 0; k < 3; k++) {
        lo[k] = org[k];
        hi[k] += 2.0 * margin;
        dims[k] = (int)std::min(64.0, std::max(1.0, ceil((hi[k] - lo[k]) / cs[k])));
        if (lo[k] + cs[k] * dims[k] < hi[k]) cs[k] = (hi[k] - lo[k]) / dims[k];      // clamped: wider cells cover the rest
    }
    const size_t n_cells = (size_t)dims[0] * dims[1] * dims[2];
    std::vector<int> count(n_cells + 1, 0);
    auto range = [&](int i, int k, int& a, int& b) {
        a = (int)floor(((double)boxes[6 * i + k] - margin - lo[k]) / cs[k]);
        b = (int)floor(((double)boxes[6 * i + 3 + k] + margin - lo[k]) / cs[k]);
        a = std::max(0, std::min(dims[k] - 1, a));
        b = std::max(0, std::min(dims[k] - 1, b));
    };
    size_t total = 0;
    for (int pass = 0; pass < 2; pass++) {
        if (pass == 1) {
            if (total > (size_t)8 * n) return false;
            for (size_t c = 0; c < n_cells; c++) {
                if (count[c] > 24) return false;
            }
            // exclusive prefix sums -> cell starts
            int run = 0;
            for (size_t c = 0; c <= n_cells; c++) {
                const int v = c < n_cells ? count[c] : 0;
                count[c] = run;
                run += v;
            }
            g.items.assign(total, 0);
        }
        std::vector<int> fill;
        if (pass == 1) fill.assign(count.begin(), count.end() - 1);
        for (int i = 0; i < n; i++) {
            int a[3], b[3];
            for (int k = 0; k < 3; k++) range(i, k, a[k], b[k]);
            for (int z = a[2]; z <= b[2]; z++)
                for (int y = a[1]; y <= b[1]; y++)
                    for (int x = a[0]; x <= b[0]; x++) {
                        const size_t c = (size_t)x + (size_t)dims[0] * ((size_t)y + (size_t)dims[1] * z);
                        if (pass == 0) {
                            count[c]++;
                            total++;
                        } else {
                            g.items[fill[c]++] = i;
                        }
                    }
        }
    }
    g.cell_start = count;
    for (int k = 0; k < 3; k++) {
        g.lo[k] = (float)lo[k];
        g.cell[k] = (float)cs[k];
        g.dims[k] = dims[k];
        g.lo_d[k] = lo[k];
        g.cell_d[k] = cs[k];
    }
    g.reg_margin_d = margin;
    g.reg_margin = (float)(0.5 * margin);     // what a ray's fattening may be: half of what the registration allowed for
    return true;
}
