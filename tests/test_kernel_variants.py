"""Every render-kernel variant the dispatcher can pick, bit for bit against the oracle, at depths that fill its level stack.

A frame is rendered by one of many separately compiled kernels: render_kernel<CAP, SBVH, FM> and its list-mode twin
(tcrt_render.cu), render_grid_kernel<CAP, FM in {0, 3}> and its twin (tcrt_render_grid.cu), hits_kernel<SBVH, FM>
(tcrt_hits.cu).  SBVH says whether the scene has a sphere BVH; FM how finite planes are swept (0 none, 1 box clusters, 2 a
finite-plane BVH, 3 linearly); CAP is the per-lane level stack, the smallest of 8, 16, 64 and 256 that holds
max_depth + 1 levels.  A slip in one combination lives only in that combination's code.

One scene builder per dispatch class puts the default camera and three lights inside a closed mirror enclosure
(reflective factor 1), so that nearly every path bounces max_depth times and stacks a record at every level.  The CPU
tests check that each builder lands in its class (the dispatch rule restated from tcrt_plan_scene's structure counts) and
that the builders cover every class; the GPU tests compare every class at the boundary depths of each CAP: band kernels
(tiled, untiled, a band from an odd column), the switches, the list kernels of adaptive frames and the hit kernels.

In every scene the last light sits 0.5e-3 inside one wall.  A shading point on that wall lies 1e-3 off it, so the light
is just below the point's tangent plane (negative cosine term) and no surface lies between them: the light is unshadowed,
and in the reference its cosineShade clamps an earlier specular highlight's local colour above 1 back to 1.  The sphere-BVH
and grid kernels skip shadow rays that cannot change the local colour and must keep tracing exactly this one.
"""
from __future__ import annotations

import math

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import assert_bit_identical
from test_hit_buffers import assert_hits_equal, hits_lib, primary_hits  # noqa: F401  (hits_lib is a fixture)

gpu = pytest.mark.gpu

# ---- the enclosure: a box of half extents HALF around CENTER, its axes rotated off the world's -------------------------------

CENTER = np.array([-1.0, -1.0, 2.5])
HALF = np.array([7.0, 7.0, 4.5])


def _rotation():
    a, b = math.radians(25.0), math.radians(12.0)
    rz = np.array([[math.cos(a), -math.sin(a), 0.0], [math.sin(a), math.cos(a), 0.0], [0.0, 0.0, 1.0]])
    rx = np.array([[1.0, 0.0, 0.0], [0.0, math.cos(b), -math.sin(b)], [0.0, math.sin(b), math.cos(b)]])
    return rx @ rz


AXES = _rotation().T          # AXES[k]: the box's k-th axis in world coordinates


def _pt(v):
    return tuple(float(x) for x in v)


def _world(local):
    """Box-local coordinates (-1..1 per axis across the box) to world coordinates."""
    return CENTER + (np.asarray(local, float) * HALF) @ AXES


def _inside_box(p, margin):
    q = (np.asarray(p, float) - CENTER) @ AXES.T
    return bool((np.abs(q) <= HALF - margin).all())


ROOM_LO, ROOM_DIMS = np.array([-8.0, -8.0, -1.0]), np.array([16.0, 16.0, 9.0])     # the axis-aligned room (box clusters)


def _inside_room(p, margin):
    p = np.asarray(p, float)
    return bool(((p >= ROOM_LO + margin) & (p <= ROOM_LO + ROOM_DIMS - margin)).all())


WALL = dict(reflective=1.0, diffuse=.4, specular=.5)


def _wall(ref, k):
    ref.setColor(.95 - .04 * k, .9, .75 + .04 * k).setReflectiveFactor(WALL["reflective"]) \
        .setDiffuseFactor(WALL["diffuse"]).setSpecularFactor(WALL["specular"])
    if k == 1:
        ref.setCheckerBoard((1, 1, 1), (.6, .7, .8), 1.5, 1.5)
    return ref


def _rotated_faces(s, tiles):
    """The six faces of the rotated box as finite planes (addFinitePlaneCorners), each tiled tiles x tiles."""
    k = 0
    for a in range(3):
        b, c = (a + 1) % 3, (a + 2) % 3
        for sgn in (-1.0, 1.0):
            centre = CENTER + sgn * HALF[a] * AXES[a]
            eb, ec = 2 * HALF[b] * AXES[b] / tiles, 2 * HALF[c] * AXES[c] / tiles
            base = centre - HALF[b] * AXES[b] - HALF[c] * AXES[c]
            for i in range(tiles):
                for j in range(tiles):
                    o = base + i * eb + j * ec
                    _wall(s.addFinitePlaneCorners(_pt(o), _pt(o + eb), _pt(o + ec)), k)
            k += 1


def _infinite_faces(s):
    """The six faces of the rotated box as infinite planes: a closed box with no finite plane."""
    for a in range(3):
        for k, sgn in enumerate((-1.0, 1.0)):
            centre = CENTER + sgn * HALF[a] * AXES[a]
            _wall(s.addInfinitePlane(_pt(centre), _pt(AXES[a]), _pt(AXES[(a + 1) % 3])), 2 * a + k)


def _room(s):
    """makeSceneBox: six axis-aligned rectangles, which the upload sweeps through box clusters."""
    for k, face in enumerate(s.makeSceneBox(_pt(ROOM_LO), _pt(ROOM_DIMS))):
        _wall(face, k)


# ---- lights and spheres ---------------------------------------------------------------------------------------------------

LIGHTS_LOCAL = [(.3, .6, .7), (-.5, .2, .75)]
GRAZE_DEPTH = 5e-4     # the last light's centre lies this far inside a wall: below the 1e-3 offset of the wall's hit points


def _lights(s, enclosure):
    """Two lights of intensity 2 and 3 inside the enclosure, then the grazing light 0.5e-3 inside its ceiling."""
    for pos, inten in zip(LIGHTS_LOCAL, (2.0, 3.0)):
        s.addSphere(_pt(_world(pos)), .15).setColor(1, .95, .9).setAsLightSource(inten)
    if enclosure == "room":
        top = ROOM_LO[2] + ROOM_DIMS[2]
        graze = (1.5, 2.0, top - GRAZE_DEPTH)
    else:
        graze = CENTER + (.2 * HALF[0]) * AXES[0] + (-.3 * HALF[1]) * AXES[1] + (HALF[2] - GRAZE_DEPTH) * AXES[2]
    s.addSphere(_pt(graze), .15).setColor(.9, 1, .95).setAsLightSource(1.5)


LATTICE = [(-2.0 + 1.0 * i, 0.0 + 1.0 * j, 1.4 + 1.2 * k) for k in range(2) for j in range(5) for i in range(5)]
FEW = [(-2.2 + 1.4 * (i % 4), -.5 + 1.5 * (i // 4), 1.2 + .5 * (i % 3)) for i in range(12)]
BIG = ((3.0, -2.5, 2.5), 1.4)    # more than 4x the median radius: no sphere grid


def _spheres(s, centres, radius):
    for n, c in enumerate(centres):
        s.addSphere(c, radius).setColor(.55 + .4 * ((n * 7) % 5) / 4, .6 + .35 * ((n * 3) % 4) / 3, .95 - .3 * (n % 3) / 2) \
            .setReflectiveFactor(1.0).setDiffuseFactor(.3).setSpecularFactor(.6)


class _PlacedRef:
    """A SceneObjectRef of a placed scene: a checkerboard's cell width and height are lengths."""

    def __init__(self, ref, scale):
        self._ref, self._scale = ref, scale

    def __getattr__(self, name):
        return getattr(self._ref, name)

    def setCheckerBoard(self, light, dark, width, height):
        self._ref.setCheckerBoard(light, dark, width * self._scale, height * self._scale)
        return self


class Placed:
    """An api.Scene built with every point x mapped to scale * x + shift (in double, rounded once to float by the API):
    radii, box dimensions and checker cells are multiplied by scale; normal and horizontal vectors stay.  It has the
    Scene calls the builders use."""

    def __init__(self, scene, scale, shift):
        self.scene, self.scale, self.shift = scene, float(scale), np.asarray(shift, float)

    def point(self, v):
        return _pt(self.scale * np.asarray(v, float) + self.shift)

    def _ref(self, ref):
        return _PlacedRef(ref, self.scale)

    def addSphere(self, origin, radius):
        return self._ref(self.scene.addSphere(self.point(origin), radius * self.scale))

    def addInfinitePlane(self, origin, normal, horizontal):
        return self._ref(self.scene.addInfinitePlane(self.point(origin), normal, horizontal))

    def addFinitePlaneCorners(self, origin, vertical_corner, horizontal_corner):
        return self._ref(self.scene.addFinitePlaneCorners(self.point(origin), self.point(vertical_corner),
                                                          self.point(horizontal_corner)))

    def makeSceneBox(self, origin, dims):
        return [self._ref(r) for r in self.scene.makeSceneBox(self.point(origin), _pt(self.scale * np.asarray(dims, float)))]

    def camera(self, cam):
        """The exported camera of `cam` under the same map."""
        c = cam.export()
        for name in ("eye", "screen_origin"):
            v = self.point(getattr(c, name)[:])
            for k in range(3):
                getattr(c, name)[k] = v[k]
        for name in ("screen_width", "screen_height", "screen_halfwidth", "screen_halfheight"):
            setattr(c, name, getattr(c, name) * self.scale)
        return c


def _scene(enclosure, spheres, big, place=None):
    """(Scene, Camera) of a builder; with place = (scale, shift): (Scene, exported camera) of it placed by Placed."""
    scene = api.Scene()
    s = scene if place is None else Placed(scene, *place)
    _lights(s, enclosure)
    if enclosure == "infinite":
        _infinite_faces(s)
    elif enclosure == "room":
        _room(s)
    else:
        _rotated_faces(s, 4 if enclosure == "tiled" else 1)
    if spheres == "few":
        _spheres(s, FEW, .45)
    elif spheres == "lattice":
        _spheres(s, LATTICE, .3)
    if big:
        _spheres(s, [BIG[0]], BIG[1])
    if place is None:
        return scene, api.Camera()
    return scene, s.camera(api.Camera())


# name -> (enclosure, spheres, one big sphere, the class the dispatcher must pick).  A class is ("render", SBVH, FM) for
# render_kernel / render_list_kernel and ("grid", 1, FM) for render_grid_kernel / its list twin; hits_kernel<SBVH, FM>
# serves both.
VARIANTS = {
    "sb0_fm0": ("infinite", "few", False, ("render", 0, 0)),
    "sb0_fm1": ("room", "few", False, ("render", 0, 1)),
    "sb0_fm2": ("tiled", "few", False, ("render", 0, 2)),
    "sb0_fm3": ("rotated", "few", False, ("render", 0, 3)),
    "sb1_fm0": ("infinite", "lattice", True, ("render", 1, 0)),
    "sb1_fm1": ("room", "lattice", True, ("render", 1, 1)),
    "sb1_fm2": ("tiled", "lattice", True, ("render", 1, 2)),
    "sb1_fm3": ("rotated", "lattice", True, ("render", 1, 3)),
    "grid_fm0": ("infinite", "lattice", False, ("grid", 1, 0)),
    "grid_fm3": ("rotated", "lattice", False, ("grid", 1, 3)),
}
NAMES = list(VARIANTS)


def build(name, place=None):
    """(Scene, Camera) of a variant, or (Scene, exported camera) placed at place = (scale, shift); keep the Scene alive
    while its flatten() is in use."""
    enclosure, spheres, big, _ = VARIANTS[name]
    return _scene(enclosure, spheres, big, place)


def dispatch_class(st):
    """The kernel tcrt_launch_render picks for a scene with these structures (tcrt_plan_scene / tcrt_scene_structures)."""
    sb = int(st["bvh_spheres"] > 0)
    n_fin = st["bvh_finite"] + st["cluster_rects"] + st["linear_finite"]
    fm = 2 if st["bvh_finite"] else 0 if n_fin == 0 else 1 if st["clusters"] else 3
    grid = st["grid_cells"] > 0 and sb and fm in (0, 3)
    return ("grid" if grid else "render", sb, fm)


def level_cap(depth):
    """The level stack of every kernel family: the smallest of 8, 16, 64, 256 that holds max_depth + 1 levels."""
    return next(c for c in (8, 16, 64, 256) if depth + 1 <= c)


# every CAP full (depth CAP - 1) and the first depth of the next CAP (depth CAP), and the deepest the API accepts
DEPTHS = [0, 7, 8, 15, 16, 63, 64, 254]
LIST_DEPTHS = [7, 8, 63, 64, 254]


# ---- no device needed ------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("name", NAMES)
def test_builder_lands_in_its_dispatch_class(name):
    s, cam = build(name)
    st = api.plan_scene(s.flatten())
    assert dispatch_class(st) == VARIANTS[name][3], st
    if name.startswith("sb1"):
        assert st["grid_cells"] == 0 and st["bvh_spheres"] >= 24, st
    if name.endswith("fm2"):
        assert st["bvh_finite"] == 96, st


def test_builders_cover_every_dispatch_class():
    """A change of a threshold (kSphereBvhMin, kFinBvhMin, the cluster or grid rules) that moves a builder out of its class
    fails here rather than silently dropping a kernel from the GPU tests."""
    got = set()
    for name in NAMES:
        s, _ = build(name)
        got.add(dispatch_class(api.plan_scene(s.flatten())))
    render = {(sb, fm) for kind, sb, fm in got if kind == "render"}
    grid = {fm for kind, _, fm in got if kind == "grid"}
    hits = {(sb, fm) for _, sb, fm in got}
    everything = {(sb, fm) for sb in (0, 1) for fm in range(4)}
    assert render == everything, sorted(render)
    assert grid == {0, 3}, sorted(grid)
    assert hits == everything, sorted(hits)


def test_depths_fill_every_level_stack():
    caps = {level_cap(d) for d in DEPTHS}
    assert caps == {8, 16, 64, 256}
    for cap in (8, 16, 64):
        assert level_cap(cap - 1) == cap and level_cap(cap) > cap
        assert {cap - 1, cap} <= set(DEPTHS)
    assert max(DEPTHS) == max(LIST_DEPTHS) == _ffi.TCRT_MAX_DEPTH


@pytest.mark.parametrize("name", NAMES)
def test_builder_keeps_paths_bouncing(name):
    """The enclosure is closed and every surface a mirror of factor 1: nearly every path reaches max_depth, so the deep
    GPU cases really stack a record at every level."""
    enclosure = VARIANTS[name][0]
    inside = _inside_room if enclosure == "room" else _inside_box
    cam = api.Camera().export()
    assert inside(cam.eye[:], .5)
    for pos in LIGHTS_LOCAL:
        assert inside(_world(pos), .5)
    s, cam = build(name)
    d = 16
    p = api.default_params(24, 16, d)
    _, cnt = O.render(s.flatten(), cam.export(), p)
    assert cnt["rays_reflect"] >= .9 * d * cnt["rays_primary"], cnt


def test_grazing_light_sits_inside_the_offset_of_its_wall():
    """The last light's centre lies between its wall and the 1e-3 offset of the wall's shading points: seen from any of
    them its cosine term is negative, yet the shadow ray never reaches the wall."""
    for name in NAMES:
        s, cam = build(name)
        flat = s.flatten()
        n = flat.n_objects
        origin = np.ctypeslib.as_array(flat.obj_origin, (n * 4,)).reshape(n, 4)[:, :3]
        graze = origin[flat.light_obj[flat.n_lights - 1]].astype(float)
        if VARIANTS[name][0] == "room":
            height = ROOM_LO[2] + ROOM_DIMS[2] - graze[2]
        else:
            height = HALF[2] - (graze - CENTER) @ AXES[2]
        assert 0 < height < 1e-3 and abs(height - GRAZE_DEPTH) < 1e-5, height


# ---- bit-exact on the GPU ------------------------------------------------------------------------------------------------

def _upload(ctx, name):
    s, cam = build(name)
    flat, c = s.flatten(), cam.export()
    ctx.upload_flat(flat, c)
    assert dispatch_class(ctx.scene_structures()) == VARIANTS[name][3], ctx.scene_structures()
    return s, flat, c


def _counters(st):
    return st.rays_primary, st.rays_shadow, st.rays_reflect


def _want_counters(cnt):
    return cnt["rays_primary"], cnt["rays_shadow"], cnt["rays_reflect"]


def frame_sizes(depth):
    """(tiled W x H, untiled W x H, band [x0, x1) of the tiled frame): W % 4 == 0 and H % 8 == 0 take the 4x8 tile claims."""
    if depth > 64:
        return (40, 32), (29, 23), (5, 31)
    return (48, 40), (45, 37), (7, 38)


def list_frame_size(depth):
    """W x H of the adaptive frames: the oracle renders 2W x 2H."""
    return (16, 12) if depth > 64 else (24, 16)


@gpu
@pytest.mark.parametrize("depth", DEPTHS)
@pytest.mark.parametrize("name", NAMES)
def test_band_kernels_match_the_oracle(gpu_ctx, name, depth):
    s, flat, c = _upload(gpu_ctx, name)
    tiled, untiled, (x0, x1) = frame_sizes(depth)
    for w, h in (tiled, untiled):
        p = api.default_params(w, h, depth)
        img, st = gpu_ctx.render(p)
        want, cnt = O.render(flat, c, p)
        what = f"{name} {w}x{h} d{depth}"
        assert_bit_identical(img, want, what)
        assert _counters(st) == _want_counters(cnt), what
    p = api.default_params(*tiled, depth)
    img, st = gpu_ctx.render(p, x0, x1)
    want, cnt = O.render(flat, c, p, x0, x1)
    what = f"{name} {tiled} columns [{x0}, {x1}) d{depth}"
    assert_bit_identical(img, want, what)
    assert _counters(st) == _want_counters(cnt), what


@gpu
@pytest.mark.parametrize("switch", ["shadows", "reflections"])
@pytest.mark.parametrize("name", NAMES)
def test_switches_match_the_oracle(gpu_ctx, name, switch):
    s, flat, c = _upload(gpu_ctx, name)
    p = api.default_params(32, 24, 16, **{switch: False})
    img, st = gpu_ctx.render(p)
    want, cnt = O.render(flat, c, p)
    what = f"{name} {switch} off"
    assert_bit_identical(img, want, what)
    assert _counters(st) == _want_counters(cnt), what


@gpu
@pytest.mark.parametrize("depth", LIST_DEPTHS)
@pytest.mark.parametrize("name", NAMES)
def test_list_kernels_match_the_oracle(gpu_ctx, name, depth):
    """Adaptive frames at contrast -1 refine every pixel through the list kernel: each pixel is the box filter of the
    oracle's 2W x 2H frame, and the call traces exactly the rays of that frame."""
    s, flat, c = _upload(gpu_ctx, name)
    ss, (w, h) = 2, list_frame_size(depth)
    p = api.default_params(w, h, depth)
    samples, cnt = O.render(flat, c, api.default_params(ss * w, ss * h, depth))
    acc = samples[0::ss, 0::ss].copy()
    for i in range(ss):
        for j in range(ss):
            if i or j:
                acc = acc + samples[i::ss, j::ss]
    want = acc / np.float32(ss * ss)
    got, _, n, st = gpu_ctx.render_adaptive(p, ss, -1)
    what = f"{name} adaptive ss={ss} d{depth}"
    assert n == w * h, what
    assert_bit_identical(got, want, what)
    assert _counters(st) == _want_counters(cnt), what


@gpu
@pytest.mark.parametrize("name", NAMES)
def test_hit_kernels_match_the_oracle(gpu_ctx, hits_lib, name):
    s, flat, c = _upload(gpu_ctx, name)
    for w, h, x0, x1 in ((32, 24, 0, 32), (27, 17, 0, 27), (32, 24, 3, 22)):
        p = api.default_params(w, h, 8)
        got, _ = gpu_ctx.hit_buffers(p, x0, x1)
        want = primary_hits(hits_lib, flat, c, p, x0, x1)
        assert_hits_equal(got, want, f"{name} {w}x{h} columns [{x0}, {x1})")
        assert (got["object"] >= 0).all(), name            # a closed enclosure: every primary ray hits something
    p = api.default_params(27, 17, 8)
    full = primary_hits(hits_lib, flat, c, p)
    rng = np.random.default_rng(len(name))
    xs = np.concatenate([[0, 26, 0, 26, 13], rng.integers(0, 27, 40)])
    zs = np.concatenate([[0, 0, 16, 16, 8], rng.integers(0, 17, 40)])
    obj, dist, normal = gpu_ctx.pick(p, xs, zs)
    want = {"object": full["object"][xs, zs], "distance": full["distance"][xs, zs], "normal": full["normal"][xs, zs]}
    assert_hits_equal({"object": obj, "distance": dist, "normal": normal}, want, f"{name} picks")
