"""Bit-exact parity for scenes moved and rescaled off the unit box, and for every far_dist the API accepts.

The culling structures (sphere BVH, box clusters, sphere grid, plane prefilter) stay exact through margins of two kinds
(DESIGN.md §4.5): relative ones that grow with the scene (the 1e-5 * max|coordinate| inflation of host boxes, the cluster
and grid margins) and absolute ones that do not (the grid walk's 2e-4 exit slack, +1e-6 in the bounding radii, the 1e-30
reciprocal clamps, the reference's own 1e-10, 1e-5 and 1e-3).  Which kind binds depends on the scene's size and on how far
it sits from the origin, and on far_dist, so every dispatch class of test_kernel_variants is rendered here

* placed: every point x of the scene and the camera mapped to scale * x + shift, at scales 2^-6, 2^6, 0.37 and 37, a
  shift of about 2^12, and, for the lattice (grid) classes, the largest shift along (1, 1, 1) at which the grid is still
  built — there the boxes' 1e-5 * |coordinate| inflation is as large as the spheres and the DDA's rounding of about
  u * |coordinate| uses up most of the grid's registration margin — and the next candidate shift, whose grid is refused;
* at every far_dist: -inf, -1, -0.1, -0, +0, a denormal, 1e-3, one that cuts through the scene, 65535, FLT_MAX, +inf and
  NaN.  A miss returns far_dist itself, so hit buffers are compared bitwise, NaN included.  At far_dist <= 0 the only
  hit left is a sphere around the ray's origin (negative distance): the grid walk must still visit the origin's cell.

The CPU tests check that each placed scene lands in its dispatch class, that its frame is not degenerate, that the
placements cover every class (the grid classes at an offset where the inflation is at least the sphere radius), that the
translated and scaled lattices register every sphere wherever it can be hit, and the oracle's own result inside a
sphere at negative far_dist, so that the GPU case cannot pass on an empty frame.
"""
from __future__ import annotations

import functools

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import api

from _util import assert_bit_identical
from test_hit_buffers import assert_hits_equal, hits_lib, primary_hits  # noqa: F401  (hits_lib is a fixture)
from test_host_api import _grid_soundness
from test_kernel_variants import NAMES, VARIANTS, build, dispatch_class
from test_occlusion import check_lights, occ_lib, scene_points  # noqa: F401  (occ_lib is a fixture)
from test_ray_batches import arbitrary_rays, oracle_hits, oracle_trace, rays_lib  # noqa: F401  (rays_lib is a fixture)
from test_ray_batches import assert_hits_equal as assert_ray_hits_equal

gpu = pytest.mark.gpu
F32 = np.float32
FLT_MAX = float(np.finfo(F32).max)
INF = float("inf")

# ---- placements --------------------------------------------------------------------------------------------------------

PLACEMENTS = {
    "scale_2^-6": (2.0 ** -6, (0.0, 0.0, 0.0)),
    "scale_2^6": (2.0 ** 6, (0.0, 0.0, 0.0)),
    "scale_0.37": (0.37, (0.0, 0.0, 0.0)),
    "scale_37": (37.0, (0.0, 0.0, 0.0)),
    "shift_2^12": (1.0, (4096.0, -0.7 * 4096.0, 0.4 * 4096.0)),
}
GRID_NAMES = [n for n in NAMES if VARIANTS[n][3][0] == "grid"]
LATTICE_RADIUS = 0.3                 # the lattice builders' sphere radius (test_kernel_variants LATTICE)
# shifts t * (1, 1, 1) searched for the grid's tightest offset, in increasing order
GRID_SHIFTS = [m * 2.0 ** k for k in range(12, 21) for m in (1.0, 1.25, 1.5, 1.75)]


def _extent(flat):
    """max |coordinate| of sphere centres and finite-plane origins, at least 1: the host boxes' inflation is 1e-5 of it."""
    sph = np.ctypeslib.as_array(flat.sphere_geom, (flat.n_spheres * 4,)).reshape(-1, 4)[:, :3]
    fin = np.ctypeslib.as_array(flat.fin_geom, (flat.n_fin_planes * 16,)).reshape(-1, 16)[:, 12:15] \
        if flat.n_fin_planes else np.zeros((0, 3), F32)
    return max(1.0, float(np.abs(sph).max(initial=0)), float(np.abs(fin).max(initial=0)))


@functools.lru_cache(maxsize=None)
def grid_offsets(name):
    """(the largest searched shift at which the lattice class keeps its grid, the next searched shift, refused), from
    tcrt_plan_scene.  Beyond the first refusal the search does not go on: the boundary is not monotone."""
    kept = None
    for t in GRID_SHIFTS:
        s, _ = build(name, (1.0, (t, t, t)))
        if api.plan_scene(s.flatten())["grid_cells"] > 0:
            kept = t
        elif kept is not None and 1e-5 * kept >= LATTICE_RADIUS:
            return kept, t
    raise AssertionError(f"{name}: no refused shift above a kept one with 1e-5 * shift >= {LATTICE_RADIUS} in {GRID_SHIFTS}")


def placement(pid, name):
    """(scale, shift) of placement id pid for the builder name."""
    if pid in PLACEMENTS:
        return PLACEMENTS[pid]
    t = grid_offsets(name)[0 if pid == "grid_tight" else 1]
    return 1.0, (t, t, t)


# (placement id, builder): every placement of every class, and the lattice classes at their tightest grid offsets
CASES = [(pid, n) for pid in PLACEMENTS for n in NAMES] + [(pid, n) for pid in ("grid_tight", "grid_refused") for n in GRID_NAMES]
CASE_IDS = [f"{pid}-{n}" for pid, n in CASES]


def expected_class(pid, name):
    """The builder's class; at the refused grid offset the same scene without its grid (the BVH kernel)."""
    kind, sb, fm = VARIANTS[name][3]
    return ("render", sb, fm) if pid == "grid_refused" else (kind, sb, fm)


def build_placed(pid, name):
    """(Scene, flat, exported camera) of a placed builder; keep the Scene alive while flat is in use."""
    s, c = build(name, placement(pid, name))
    return s, s.flatten(), c


def placed_params(pid, name, w, h, depth):
    """A scaled-up scene is rendered at far_dist = +inf: the default 65535 could hide what lies beyond it."""
    p = api.default_params(w, h, depth)
    if placement(pid, name)[0] > 1.0:
        p.far_dist = INF
    return p


DEPTHS = (7, 16)          # one full level stack of 8, and one of 64


def frame_size(depth):
    """A tiled frame (W % 4 == 0, H % 8 == 0) at the shallow depth, an untiled one at the deep depth."""
    return (48, 40) if depth < 8 else (45, 37)


# ---- far_dist --------------------------------------------------------------------------------------------------------

FAR_DISTS = [-INF, -1.0, -0.1, -0.0, 0.0, 1e-40, 1e-3, 6.0, 65535.0, FLT_MAX, INF, float("nan")]
FAR_IDS = ["-inf", "-1", "-0.1", "-0", "+0", "denormal", "1e-3", "6", "65535", "FLT_MAX", "+inf", "nan"]
assert F32(1e-40) != 0 and abs(F32(1e-40)) < np.finfo(F32).tiny


def far_params(w, h, depth, far):
    p = api.default_params(w, h, depth)
    p.far_dist = far
    return p


def inside_sphere_scene():
    """The grid scene with the camera inside a lattice sphere (test_sphere_grid_edge_cases[inside_sphere])."""
    from test_adaptive_frames import _inside_sphere_scene

    return _inside_sphere_scene()


def _non_null(img, p):
    return int((img != np.array(p.null_color[:], F32)).any(-1).sum())


# ---- no device needed ------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("pid,name", CASES, ids=CASE_IDS)
def test_placed_builder_lands_in_its_dispatch_class(pid, name):
    s, flat, _ = build_placed(pid, name)
    st = api.plan_scene(flat)
    assert dispatch_class(st) == expected_class(pid, name), st
    if pid == "grid_refused":
        assert st["grid_cells"] == 0 and st["bvh_spheres"] >= 24, st


@pytest.mark.parametrize("pid,name", CASES, ids=CASE_IDS)
def test_placed_frames_are_not_degenerate(pid, name):
    """The enclosure stays closed under every placement: nearly every pixel sees a surface and nearly every path reaches
    max_depth, so the GPU cases compare real frames at every level.  At the grid offsets (2^16 and beyond) the corners
    of the rotated walls round to a 2^-7 lattice and leave slits through which some paths escape."""
    s, flat, c = build_placed(pid, name)
    d = 16
    p = placed_params(pid, name, 24, 16, d)
    img, cnt = O.render(flat, c, p)
    seen, bouncing = (.8, .4) if pid.startswith("grid") else (.95, .9)
    assert _non_null(img, p) >= seen * p.width * p.height, (pid, name)
    assert cnt["rays_reflect"] >= bouncing * d * cnt["rays_primary"], cnt


def test_placements_cover_every_dispatch_class():
    """Every class appears among the placed scenes, and the grid classes appear at an offset where the grid is built and
    the 1e-5 * |coordinate| inflation of the host boxes is at least the sphere radius."""
    got = set()
    for pid, name in CASES:
        s, flat, _ = build_placed(pid, name)
        st = api.plan_scene(flat)
        got.add(dispatch_class(st))
        if pid == "grid_tight":
            assert st["grid_cells"] > 0 and 1e-5 * _extent(flat) >= LATTICE_RADIUS, (name, _extent(flat), st)
    want = {("render", sb, fm) for sb in (0, 1) for fm in range(4)} | {("grid", 1, 0), ("grid", 1, 3)}
    assert got == want, sorted(got)


@pytest.mark.parametrize("name", GRID_NAMES)
def test_grid_offsets_bracket_the_grid(name):
    kept, refused = grid_offsets(name)
    assert kept < refused and 1e-5 * kept >= LATTICE_RADIUS
    for t, grid in ((kept, True), (refused, False)):
        s, _ = build(name, (1.0, (t, t, t)))
        assert (api.plan_scene(s.flatten())["grid_cells"] > 0) == grid, (name, t)


@pytest.mark.parametrize("pid", list(PLACEMENTS) + ["grid_tight"])
@pytest.mark.parametrize("name", GRID_NAMES)
def test_placed_lattices_register_every_sphere(pid, name):
    """DESIGN.md §4.5 (i) on the translated and scaled lattices: every point of a sphere and of its shell out to the grid's
    margin lies in a cell that lists the sphere."""
    s, flat, _ = build_placed(pid, name)
    plan = api.plan_scene(flat)
    assert plan["grid_cells"] > 0
    n = flat.n_spheres
    geom = np.ctypeslib.as_array(flat.sphere_geom, (n * 4,)).reshape(n, 4)
    objs = np.ctypeslib.as_array(flat.sphere_obj, (n,))
    info = np.ctypeslib.as_array(flat.obj_info, (flat.n_objects * 4,)).reshape(-1, 4)
    spheres = [(int(o), g[:3].astype(float), float(np.sqrt(g[3]))) for g, o in zip(geom, objs) if info[o, 2] == 0]
    assert len(spheres) == plan["bvh_spheres"]
    _grid_soundness(flat, spheres, 17)


@pytest.mark.parametrize("far", FAR_DISTS, ids=FAR_IDS)
def test_oracle_inside_a_sphere_at_every_far_dist(far):
    """The reference keeps a hit while dist < far_dist.  From inside a sphere its distance is negative: at far_dist in
    (-1, 0] nearly every pixel still sees the enclosing sphere; at -1 and below, and at NaN, nothing is hit."""
    s, c = inside_sphere_scene()
    p = far_params(32, 24, 4, far)
    img, cnt = O.render(s.flatten(), c, p)
    seen = _non_null(img, p)
    if far != far or far <= -1.0:
        assert seen == 0 and cnt["rays_shadow"] == 0 and cnt["rays_reflect"] == 0, (far, seen, cnt)
    elif far <= 0.0:
        assert seen >= 700, (far, seen)
    else:
        assert seen > 0


# ---- bit-exact on the GPU ------------------------------------------------------------------------------------------------

def _counters(st):
    return st.rays_primary, st.rays_shadow, st.rays_reflect


def _want_counters(cnt):
    return cnt["rays_primary"], cnt["rays_shadow"], cnt["rays_reflect"]


def check_frame(ctx, flat, c, p, what):
    img, st = ctx.render(p)
    want, cnt = O.render(flat, c, p)
    assert_bit_identical(img, want, what)
    assert _counters(st) == _want_counters(cnt), what
    return want


@gpu
@pytest.mark.parametrize("pid,name", CASES, ids=CASE_IDS)
def test_placed_scenes_match_the_oracle(gpu_ctx, hits_lib, rays_lib, occ_lib, pid, name):
    s, flat, c = build_placed(pid, name)
    gpu_ctx.upload_flat(flat, c)
    assert dispatch_class(gpu_ctx.scene_structures()) == expected_class(pid, name), gpu_ctx.scene_structures()
    for depth in DEPTHS:
        check_frame(gpu_ctx, flat, c, placed_params(pid, name, *frame_size(depth), depth), f"{pid} {name} d{depth}")
    p = placed_params(pid, name, 27, 17, 8)
    got, _ = gpu_ctx.hit_buffers(p)
    assert_hits_equal(got, primary_hits(hits_lib, flat, c, p), f"{pid} {name} hit buffers")
    rng = np.random.default_rng(CASES.index((pid, name)))
    o, d, _ = arbitrary_rays(gpu_ctx, flat, c, name, rng)
    p = placed_params(pid, name, 1, 1, 0)
    got_h, n_bad, _ = gpu_ctx.intersect_rays(p, o, d)
    want_h, w_bad = oracle_hits(rays_lib, flat, p, o, d)
    assert n_bad == w_bad
    assert_ray_hits_equal(got_h, want_h, f"{pid} {name} intersect_rays")
    check_lights(gpu_ctx, occ_lib, flat, scene_points(gpu_ctx, occ_lib, flat, c, rng), f"{pid} {name} occluded_lights")


@gpu
@pytest.mark.parametrize("name", NAMES)
def test_every_far_dist_in_every_dispatch_class(gpu_ctx, hits_lib, name):
    s, cam = build(name)
    flat, c = s.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    assert dispatch_class(gpu_ctx.scene_structures()) == VARIANTS[name][3]
    for far, fid in zip(FAR_DISTS, FAR_IDS):
        for depth in (0, 8):
            check_frame(gpu_ctx, flat, c, far_params(32, 24, depth, far), f"{name} far {fid} d{depth}")
        p = far_params(27, 17, 0, far)
        got, _ = gpu_ctx.hit_buffers(p)
        assert_hits_equal(got, primary_hits(hits_lib, flat, c, p), f"{name} far {fid} hit buffers")


@gpu
@pytest.mark.parametrize("far", FAR_DISTS, ids=FAR_IDS)
def test_every_far_dist_inside_a_grid_sphere(gpu_ctx, hits_lib, far):
    """The camera inside a lattice sphere of a grid scene: at far_dist in (-1, 0] the enclosing sphere's negative
    distance still wins, and the grid walk has to visit the origin's cell to find it."""
    s, c = inside_sphere_scene()
    flat = s.flatten()
    gpu_ctx.upload_flat(flat, c)
    assert gpu_ctx.scene_structures()["grid_cells"] > 0
    for depth in (0, 4):
        check_frame(gpu_ctx, flat, c, far_params(32, 24, depth, far), f"inside_sphere far {far} d{depth}")
    p = far_params(32, 24, 0, far)
    got, _ = gpu_ctx.hit_buffers(p)
    assert_hits_equal(got, primary_hits(hits_lib, flat, c, p), f"inside_sphere far {far} hit buffers")


@gpu
def test_every_far_dist_in_ray_batches(gpu_ctx, rays_lib):
    """Caller-supplied rays on synth256 (grid): random origins, surface points, origins inside spheres, far origins."""
    from _util import make_scene

    s, cam = make_scene("synth256")
    flat, c = s.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    assert gpu_ctx.scene_structures()["grid_cells"] > 0
    o, d, _ = arbitrary_rays(gpu_ctx, flat, c, "synth256", np.random.default_rng(3))
    for far, fid in zip(FAR_DISTS, FAR_IDS):
        p = far_params(1, 1, 5, far)
        want, w_bad, cnt = oracle_trace(rays_lib, flat, p, o, d)
        got, g_bad, st = gpu_ctx.trace_rays(p, o, d)
        assert g_bad == w_bad == 0
        assert_bit_identical(got.reshape(-1, 1, 3), want.reshape(-1, 1, 3), f"synth256 rays far {fid}")
        assert _counters(st) == _want_counters(cnt), fid
        want_h, _ = oracle_hits(rays_lib, flat, p, o, d)
        got_h, _, _ = gpu_ctx.intersect_rays(p, o, d)
        assert_ray_hits_equal(got_h, want_h, f"synth256 rays far {fid}")
