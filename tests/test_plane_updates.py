"""Moving planes (tcrt_update_planes): new geometry, normal and origin rows for finite and infinite planes of the resident
scene, applied on the GPU by scattering the rows, refitting the finite-plane BVH and the box clusters' hulls (or dropping
the clusters), and rewriting the light table.  After an update every call that reads the scene must return, bit for bit,
what it returns after a fresh tcrt_upload_scene of the scene with those rows replaced, and, for small frames, what the
oracle renders of it.

Moved rows come from the reference's own constructors: the moved plane is built in a scratch Scene, flattened, and its rows
spliced into a copy of the original flattened scene at the object's slot."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import assert_bit_identical, bits
from test_kernel_variants import (ROOM_DIMS, ROOM_LO, VARIANTS, _infinite_faces, _lights, _room, _rotated_faces,
                                  _spheres, BIG, FEW, LATTICE, dispatch_class)
from test_material_edits import random_edit
from test_occlusion import occ_lib, oracle_lights  # noqa: F401  (occ_lib is a fixture)
from test_scene_updates import _class, counters, fresh, geom_of, inward_jitter, light_spheres, moved_flat

gpu = pytest.mark.gpu
F32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HIT_NAMES = ("object", "distance", "normal")
PLANE_NAMES = list(VARIANTS)   # every class has planes: infinite (fm0), a room (fm1), tiles (fm2), a rotated box (fm3)


@pytest.fixture(scope="module")
def ref_ctx():
    """A second context for the fresh uploads the updated one is compared with."""
    ctx = api.Context([0])
    yield ctx
    ctx.close()


# ---- scenes whose plane constructions are known ---------------------------------------------------------------------------

class Recorder:
    """An api.Scene that remembers how each plane was constructed: object index -> (kind, args), kind "inf" (origin, normal,
    horizontal), "corners" (origin, vertical corner, horizontal corner) or "box" (origin, dims, face).  subst: object index
    -> a construction of the same kind to build instead (a box's six faces only together, from one new origin)."""

    def __init__(self, subst=None):
        self.scene = api.Scene()
        self.calls = {}
        self.subst = subst or {}

    def _args(self, kind, args):
        k, a = self.subst.get(self.scene.getObjectCount(), (kind, args))
        assert k == kind
        return a

    def addSphere(self, origin, radius):
        return self.scene.addSphere(origin, radius)

    def addInfinitePlane(self, origin, normal, horizontal):
        r = self.scene.addInfinitePlane(*self._args("inf", (origin, normal, horizontal)))
        self.calls[r.index] = ("inf", (origin, normal, horizontal))
        return r

    def addFinitePlaneCorners(self, origin, vertical_corner, horizontal_corner):
        r = self.scene.addFinitePlaneCorners(*self._args("corners", (origin, vertical_corner, horizontal_corner)))
        self.calls[r.index] = ("corners", (origin, vertical_corner, horizontal_corner))
        return r

    def makeSceneBox(self, origin, dims):
        first = self.scene.getObjectCount()
        faces = [self.subst.get(first + k) for k in range(6)]
        new_origin, new_dims = origin, dims
        if any(faces):
            assert all(f and f[1][:2] == faces[0][1][:2] for f in faces), "a box moves as a whole"
            new_origin, new_dims = faces[0][1][:2]
        refs = self.scene.makeSceneBox(new_origin, new_dims)
        for k, r in enumerate(refs):
            self.calls[r.index] = ("box", (origin, dims, k))
        return refs


def build(name, subst=None):
    """(Recorder, Camera) of a variant of test_kernel_variants, the same scene object for object; with subst, the
    constructions of those objects replaced."""
    enclosure, spheres, big, _ = VARIANTS[name]
    s = Recorder(subst)
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
    return s, api.Camera()


def construct(call):
    """The (geom, normals, origin) rows of one plane construction, built by the reference's constructors."""
    kind, args = call
    s = api.Scene()
    if kind == "inf":
        s.addInfinitePlane(*args)
        k = 0
    elif kind == "corners":
        s.addFinitePlaneCorners(*args)
        k = 0
    else:
        s.makeSceneBox(args[0], args[1])
        k = args[2]
    return tuple(a[0] for a in api.plane_rows(s.flatten(), [k]))


def _rows(flat, name, width, count, dtype=F32):
    if count == 0:
        return np.zeros((0, width), dtype)
    return np.ctypeslib.as_array(getattr(flat, name), (count * width,)).reshape(count, width).astype(dtype)


class Move:
    """Rows for update_planes, and the spliced copy of a flattened scene they must be indistinguishable from."""

    def __init__(self, objects, geom, normals, origin):
        self.objects = np.asarray(objects, np.int32)
        self.geom = np.ascontiguousarray(geom, F32).reshape(-1, 16)
        self.normals = np.ascontiguousarray(normals, F32).reshape(-1, 8)
        self.origin = np.ascontiguousarray(origin, F32).reshape(-1, 4)

    @classmethod
    def of(cls, calls):
        """calls: object index -> construction of its moved plane."""
        objs = sorted(calls)
        rows = [construct(calls[o]) for o in objs]
        return cls(objs, [r[0] for r in rows], [r[1] for r in rows], [r[2] for r in rows])

    def apply(self, ctx):
        return ctx.update_planes(self.objects, self.geom, self.normals, self.origin)

    def flat(self, flat):
        m = _ffi.TcrtScene.from_buffer_copy(bytes(flat))
        n = flat.n_objects
        info = _rows(flat, "obj_info", 4, n, np.int32)
        fin = _rows(flat, "fin_geom", 16, flat.n_fin_planes).copy()
        inf = _rows(flat, "inf_geom", 16, flat.n_inf_planes).copy()
        normals = _rows(flat, "obj_normals", 8, n).copy()
        origin = _rows(flat, "obj_origin", 4, n).copy()
        for i, o in enumerate(self.objects):
            (fin if info[o, 0] == 1 else inf)[info[o, 1]] = self.geom[i]
            normals[o] = self.normals[i]
            origin[o] = self.origin[i]
        m.fin_geom = fin.ctypes.data_as(_ffi.c_float_p) if len(fin) else None
        m.inf_geom = inf.ctypes.data_as(_ffi.c_float_p) if len(inf) else None
        m.obj_normals = normals.ctypes.data_as(_ffi.c_float_p)
        m.obj_origin = origin.ctypes.data_as(_ffi.c_float_p)
        m._keep = (fin, inf, normals, origin, flat)
        return m


# ---- rigid moves of constructions ---------------------------------------------------------------------------------------

def _rot(axis, deg):
    a = np.asarray(axis, float) / np.linalg.norm(axis)
    t = math.radians(deg)
    k = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    return np.eye(3) + math.sin(t) * k + (1 - math.cos(t)) * k @ k


def _t(v):
    return tuple(float(x) for x in v)


def rigid(call, shift=(0, 0, 0), rot=None, pivot=None):
    """The construction moved rigidly: rotated by rot about pivot (default its first point), then shifted.  A box face
    (makeSceneBox: axis-aligned) is only shifted."""
    kind, args = call
    shift = np.asarray(shift, float)
    if kind == "box":
        return ("box", (_t(np.asarray(args[0]) + shift), args[1], args[2]))
    r = np.eye(3) if rot is None else rot
    p0 = np.asarray(args[0], float) if pivot is None else np.asarray(pivot, float)
    pt = lambda v: _t(r @ (np.asarray(v, float) - p0) + p0 + shift)   # noqa: E731
    if kind == "inf":
        return ("inf", (pt(args[0]), _t(r @ np.asarray(args[1], float)), _t(r @ np.asarray(args[2], float))))
    return ("corners", tuple(pt(v) for v in args))


def corners_of_face(flat, o):
    """A finite plane's rows as a corners construction (its origin, origin + v*v_dist, origin + h*h_dist)."""
    g = api.plane_rows(flat, [o])[0][0].astype(float)
    po = g[12:15]
    return ("corners", (_t(po), _t(po + g[8:11] * g[11]), _t(po + g[4:7] * g[7])))


def face_axis(call):
    g = construct(call)[0]
    a = int(np.argmax(np.abs(g[:3])))
    return a, float(np.sign(g[a]) * g[3])


def plane_objects(rec):
    return sorted(rec.calls)


def variant_moves(name, rec, flat, rng):
    """[(what, {object: moved construction}, class the update must leave)]: random rigid moves of plane subsets."""
    calls = rec.calls
    planes = plane_objects(rec)
    enclosure = VARIANTS[name][0]
    cls = VARIANTS[name][3]
    steps = []
    if enclosure == "room":
        steps.append(("room translated", {o: rigid(calls[o], shift=(.3, -.2, .15)) for o in planes}, cls))
        # one face moved inwards along its normal: the cluster's hull stays the union, no longer tight on that face
        far = max(planes, key=lambda o: face_axis(calls[o]) if face_axis(calls[o])[0] == 0 else (-1, 0))
        a, _ = face_axis(calls[far])
        shift = np.zeros(3)
        shift[a] = -1.5
        steps.append(("one face inwards", {far: rigid(calls[far], shift=shift)}, cls))
    elif enclosure == "tiled":
        sub = sorted(rng.choice(planes, 20, replace=False))
        moves = {o: rigid(calls[o], shift=rng.normal(0, .05, 3), rot=_rot(rng.normal(0, 1, 3), rng.normal(0, 2)))
                 for o in sub}
        steps.append(("tiles jittered", moves, cls))
        steps.append(("one tile far away", {planes[5]: rigid(calls[planes[5]], shift=(40, -25, 30))}, cls))
    elif enclosure == "infinite":
        sub = planes[:2] + planes[4:5]          # includes the checker wall (k == 1)
        steps.append(("planes tilted", {o: rigid(calls[o], rot=_rot(rng.normal(0, 1, 3), 4 + 3 * i))
                                        for i, o in enumerate(sub)}, cls))
    else:   # the rotated box: its six walls
        moves = {o: rigid(calls[o], shift=rng.normal(0, .1, 3), rot=_rot(rng.normal(0, 1, 3), rng.normal(0, 1.5)))
                 for o in planes}
        steps.append(("walls moved", moves, cls))
    return steps


def frame_pair(ctx, ref, mflat, cam, p, what, oracle=False):
    img, st = ctx.render(p)
    img = img.copy()
    fresh(ref, mflat, cam)
    want, wst = ref.render(p)
    assert_bit_identical(img, want, f"{what} vs fresh upload")
    if _class(ctx) == _class(ref):   # the same kernel: the same rays
        assert counters(st) == counters(wst), what
    if oracle:
        o, cnt = O.render(mflat, cam, p)
        assert_bit_identical(img, o, f"{what} vs oracle")
        assert counters(st) == (cnt["rays_primary"], cnt["rays_shadow"], cnt["rays_reflect"]), what
    return img


def cluster_drop_moves(rec, flat):
    """A room face turned off-axis, and one turned onto another normal axis: both drop the clusters."""
    calls = rec.calls
    face = plane_objects(rec)[0]
    corners = corners_of_face(flat, face)
    centre = np.mean([np.asarray(v, float) for v in corners[1]], axis=0)
    a, _ = face_axis(calls[face])
    inplane = np.zeros(3)
    inplane[(a + 1) % 3] = 1
    off_axis = rigid(corners, rot=_rot(inplane, 3.0), pivot=centre)
    swap = rigid(corners, rot=_rot(inplane, 90.0), pivot=centre)
    return [("face off-axis", {face: off_axis}), ("face on another axis", {face: swap})]


def shell_scene(light_plane_inside=True):
    """The room of the fm1 variants with its sphere lights, and one small finite-plane light inside it."""
    s = Recorder()
    _lights(s, "room")
    _room(s)
    _spheres(s, FEW, .45)
    o = np.array([1.0, -2.0, 5.0])
    s.addFinitePlaneCorners(_t(o), _t(o + (0, .5, 0)), _t(o + (.5, 0, 0))).setColor(1, 1, .9).setAsLightSource(2.0)
    return s, api.Camera()


# ---- without a GPU ---------------------------------------------------------------------------------------------------------

def test_entry_point_is_exported():
    assert hasattr(_ffi.load(), "tcrt_update_planes")


def test_entry_point_refuses_a_null_context():
    lib = _ffi.load()
    objs = np.zeros(1, np.int32)
    rows = np.zeros((1, 16), F32)
    p, r = objs.ctypes.data_as(C.c_void_p), rows.ctypes.data_as(C.c_void_p)
    assert lib.tcrt_update_planes(None, 1, p, r, r, r, None) == _ffi.TCRT_ERR_INVALID


def test_plane_rows_are_the_flattened_scene():
    s = api.Scene()
    s.addSphere((0, 0, 0), 1)
    s.addFinitePlaneCorners((1, 2, 3), (1, 5, 3), (4, 2, 3.5))
    s.addInfinitePlane((0, 0, -1), (0, .1, 1), (1, 0, 0)).setCheckerBoard((1, 1, 1), (0, 0, 0), 1, 1)
    s.makeSceneBox((-1, -1, -1), (2, 3, 4))
    s.addFinitePlaneAxes((0, 1, 0), (0, 0, 1), (1, 0, 0), 2.0, 3.0).setAsLightSource(1.5)
    flat = s.flatten()
    objs = [8, 2, 1, 5]
    geom, normals, origin = api.plane_rows(flat, objs)
    assert geom.dtype == normals.dtype == origin.dtype == F32
    assert geom.shape == (4, 16) and normals.shape == (4, 8) and origin.shape == (4, 4)
    fin = _rows(flat, "fin_geom", 16, flat.n_fin_planes)
    inf = _rows(flat, "inf_geom", 16, flat.n_inf_planes)
    info = _rows(flat, "obj_info", 4, flat.n_objects, np.int32)
    for i, o in enumerate(objs):
        want = (fin if info[o, 0] == 1 else inf)[info[o, 1]]
        assert (bits(geom[i]) == bits(want)).all(), o
    assert (bits(normals) == bits(_rows(flat, "obj_normals", 8, flat.n_objects)[objs])).all()
    assert (bits(origin) == bits(_rows(flat, "obj_origin", 4, flat.n_objects)[objs])).all()
    with pytest.raises(AssertionError):
        api.plane_rows(flat, [0])     # a sphere


def _splice_cases():
    """(name, what, recorder, flattened scene, Move, class a fresh upload of the spliced scene gets)."""
    rng = np.random.default_rng(1)
    for name in PLANE_NAMES:
        rec, _ = build(name)
        flat = rec.scene.flatten()
        for what, calls, _ in variant_moves(name, rec, flat, rng):
            yield name, what, rec, flat, calls


ARRAYS = (("sphere_geom", 4, "n_spheres"), ("fin_geom", 16, "n_fin_planes"), ("inf_geom", 16, "n_inf_planes"),
          ("obj_surface", 4, "n_objects"), ("obj_material", 4, "n_objects"), ("obj_origin", 4, "n_objects"),
          ("obj_normals", 8, "n_objects"), ("obj_info", 4, "n_objects"), ("textures", 8, "n_textures"))


def assert_same_flat(a, b, what):
    for name in ("n_objects", "n_spheres", "n_fin_planes", "n_inf_planes", "n_lights", "n_textures"):
        assert getattr(a, name) == getattr(b, name), f"{what} {name}"
    for name, width, count in ARRAYS:
        n = getattr(a, count) * width
        if n:
            x = np.ctypeslib.as_array(C.cast(getattr(a, name), C.POINTER(C.c_uint32)), (n,))
            y = np.ctypeslib.as_array(C.cast(getattr(b, name), C.POINTER(C.c_uint32)), (n,))
            assert (x == y).all(), f"{what} {name}"


def test_spliced_flat_is_a_fresh_build():
    """Move.flat of a flattened scene is, byte for byte, the flattened scene built with the moved constructions."""
    rng = np.random.default_rng(1)
    checked = 0
    for name in PLANE_NAMES:
        rec, _ = build(name)
        flat = rec.scene.flatten()
        for what, calls, _ in variant_moves(name, rec, flat, rng):
            if what == "one face inwards":   # one face of a makeSceneBox: no constructor builds it alone
                continue
            moved, _ = build(name, calls)
            assert_same_flat(Move.of(calls).flat(flat), moved.scene.flatten(), f"{name} {what}")
            checked += 1
    assert checked >= 6


def test_spliced_room_is_the_moved_room():
    """A whole room moved: the spliced flat equals the flat of the room built at its new place."""
    s0, s1 = Recorder(), Recorder()
    _lights(s0, "room")
    _room(s0)
    _lights(s1, "room")
    s1.makeSceneBox(_t(ROOM_LO + (.3, -.2, .15)), _t(ROOM_DIMS))
    f0, f1 = s0.scene.flatten(), s1.scene.flatten()
    calls = {o: rigid(s0.calls[o], shift=(.3, -.2, .15)) for o in s0.calls}
    m = Move.of(calls).flat(f0)
    for name, width, count in (("fin_geom", 16, f0.n_fin_planes), ("obj_normals", 8, f0.n_objects),
                               ("obj_origin", 4, f0.n_objects)):
        a = np.ctypeslib.as_array(getattr(m, name), (width * count,))
        b = np.ctypeslib.as_array(getattr(f1, name), (width * count,))
        assert (a.view(np.uint32) == b.view(np.uint32)).all(), name


def test_spliced_flats_land_in_their_classes():
    rng = np.random.default_rng(1)
    for name in PLANE_NAMES:
        rec, _ = build(name)
        flat = rec.scene.flatten()
        for what, calls, cls in variant_moves(name, rec, flat, rng):
            got = dispatch_class(api.plan_scene(Move.of(calls).flat(flat)))
            if what == "one tile far away":
                assert got[2] == 2, (name, what, got)
            else:
                assert got == cls, (name, what, got)
    for name in ("sb0_fm1", "sb1_fm1"):
        rec, _ = build(name)
        flat = rec.scene.flatten()
        off, _ = cluster_drop_moves(rec, flat)
        assert dispatch_class(api.plan_scene(Move.of(off[1]).flat(flat)))[2] == 3, name   # five rectangles: no clusters


# ---- on the GPU ------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("depth", [0, 8, 64])
@pytest.mark.parametrize("name", PLANE_NAMES)
def test_every_plane_class(gpu_ctx, ref_ctx, name, depth):
    rec, cam = build(name)
    flat, c = rec.scene.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    rng = np.random.default_rng(200 + depth + len(name))
    p = api.default_params(32, 24, depth)
    for what, calls, cls in variant_moves(name, rec, flat, rng):
        mv = Move.of(calls)
        st = mv.apply(gpu_ctx)
        assert counters(st) == (0, 0, 0) and st.gpu_launches >= 1
        assert _class(gpu_ctx) == cls, f"{name} {what}: the update changed the dispatch class"
        frame_pair(gpu_ctx, ref_ctx, mv.flat(flat), c, p, f"{name} {what} d{depth}", oracle=depth <= 8)
        flat = mv.flat(flat)   # the next move starts from this scene


@gpu
@pytest.mark.parametrize("name", ["sb0_fm1", "sb1_fm1"])
def test_cluster_drop(gpu_ctx, ref_ctx, name):
    rec, cam = build(name)
    flat, c = rec.scene.flatten(), cam.export()
    p = api.default_params(40, 32, 8)
    for what, calls in cluster_drop_moves(rec, flat):
        gpu_ctx.upload_flat(flat, c)
        assert gpu_ctx.scene_structures()["clusters"] > 0
        mv = Move.of(calls)
        mv.apply(gpu_ctx)
        st = gpu_ctx.scene_structures()
        assert st["clusters"] == 0 and st["cluster_rects"] == 0, (what, st)
        assert _class(gpu_ctx)[2] == 3, what
        frame_pair(gpu_ctx, ref_ctx, mv.flat(flat), c, p, f"{name} {what}", oracle=True)
        # the dropped clusters stay dropped; further moves keep parity
        back = Move.of({o: rec.calls[o] for o in calls})
        back.apply(gpu_ctx)
        assert gpu_ctx.scene_structures()["clusters"] == 0
        frame_pair(gpu_ctx, ref_ctx, flat, c, p, f"{name} {what}, back")


@gpu
def test_shell_masks(gpu_ctx, ref_ctx):
    """A light that was inside the room ends up outside when the room moves, then inside again; a finite-plane light
    moved out through a wall and back.  A stale inside mask would skip the walls between the light and a shading point."""
    rec, cam = shell_scene()
    flat, c = rec.scene.flatten(), cam.export()
    p = api.default_params(48, 32, 8)
    gpu_ctx.upload_flat(flat, c)
    room = [o for o, (kind, _) in rec.calls.items() if kind == "box"]
    light = [o for o, (kind, _) in rec.calls.items() if kind == "corners"][0]
    up = Move.of({o: rigid(rec.calls[o], shift=(0, 0, 8.5)) for o in room})    # the room's floor above the lights
    up.apply(gpu_ctx)
    frame_pair(gpu_ctx, ref_ctx, up.flat(flat), c, p, "room moved off the lights", oracle=True)
    back = Move.of({o: rec.calls[o] for o in room})
    back.apply(gpu_ctx)
    frame_pair(gpu_ctx, ref_ctx, flat, c, p, "room back", oracle=True)
    out = Move.of({light: rigid(rec.calls[light], shift=(0, 0, 4.5))})        # through the ceiling
    out.apply(gpu_ctx)
    m = out.flat(flat)
    assert _rows(m, "obj_origin", 4, m.n_objects)[light, 2] > ROOM_LO[2] + ROOM_DIMS[2]
    frame_pair(gpu_ctx, ref_ctx, m, c, p, "plane light outside", oracle=True)
    Move.of({light: rec.calls[light]}).apply(gpu_ctx)
    frame_pair(gpu_ctx, ref_ctx, flat, c, p, "plane light back inside", oracle=True)


@gpu
@pytest.mark.parametrize("name", ["sb1_fm3", "grid_fm3"])
def test_ext_growth(gpu_ctx, ref_ctx, name):
    """A wall moved to about 1000x the scene's extent: the spheres' boxes are widened in the same call."""
    rec, cam = build(name)
    flat, c = rec.scene.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    before = _class(gpu_ctx)
    wall = plane_objects(rec)[2]
    mv = Move.of({wall: rigid(rec.calls[wall], shift=(9000, -6000, 4000))})
    st = mv.apply(gpu_ctx)
    assert st.gpu_launches >= 3        # the sphere launches ran too
    after = _class(gpu_ctx)
    assert after[1:] == before[1:] and after[0] in (before[0], "render"), (before, after)
    assert (gpu_ctx.scene_structures()["grid_cells"] > 0) == (after[0] == "grid")
    p = api.default_params(40, 32, 8)
    m = mv.flat(flat)
    frame_pair(gpu_ctx, ref_ctx, m, c, p, f"{name} wall far away", oracle=True)
    # a sphere update after it boxes with the planes' new extent
    g = inward_jitter(geom_of(m), np.random.default_rng(3), .01, fixed=light_spheres(m))
    gpu_ctx.update_spheres(g)
    frame_pair(gpu_ctx, ref_ctx, moved_flat(m, g), c, p, f"{name} spheres moved after the wall")
    Move.of({wall: rec.calls[wall]}).apply(gpu_ctx)
    frame_pair(gpu_ctx, ref_ctx, moved_flat(flat, g), c, p, f"{name} wall back")


@gpu
@pytest.mark.parametrize("name", ["sb1_fm1", "sb0_fm2", "grid_fm0"])
def test_every_other_reader(gpu_ctx, ref_ctx, occ_lib, name):
    from test_views import three_views

    rec, cam = build(name)
    flat, c = rec.scene.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    rng = np.random.default_rng(4)
    p = api.default_params(40, 32, 8)
    xs, zs = rng.integers(0, 40, 30), rng.integers(0, 32, 30)
    g = geom_of(flat)
    pts = np.concatenate([g[:, :3] + F32(.5), rng.uniform(-6, 6, (500, 3)).astype(F32)]).astype(F32)
    o = np.array(c.eye[:], F32)
    d = api.normalize_like_reference(rng.normal(0, 1, (400, 3)).astype(F32))
    t = rng.uniform(.5, 20, 400).astype(F32)
    what, calls, _ = variant_moves(name, rec, flat, rng)[0]
    mv = Move.of(calls)
    mv.apply(gpu_ctx)
    m = mv.flat(flat)
    fresh(ref_ctx, m, c)
    a, _ = gpu_ctx.render_rgb8(p)
    b, _ = ref_ctx.render_rgb8(p)
    assert (a == b).all(), "rgb8"
    a, _ = gpu_ctx.render_ss(p, 2)
    b, _ = ref_ctx.render_ss(p, 2)
    assert_bit_identical(a.copy(), b, "ss=2")
    a, ma, na, _ = gpu_ctx.render_adaptive(p, 2, 8, mask=np.zeros((40, 32), np.uint8))
    a, ma = a.copy(), ma.copy()
    b, mb, nb, _ = ref_ctx.render_adaptive(p, 2, 8, mask=np.zeros((40, 32), np.uint8))
    assert na == nb and (ma == mb).all()
    assert_bit_identical(a, b, "adaptive")
    va, sa = gpu_ctx.render_views(p, three_views(c))
    va = va.copy()
    vb, sb = ref_ctx.render_views(p, three_views(c))
    for v in range(3):
        assert_bit_identical(va[v], vb[v], f"view {v}")
    assert counters(sa) == counters(sb)
    ra, bad_a, sta = gpu_ctx.trace_rays(p, o, d)
    ra = ra.copy()
    rb, bad_b, stb = ref_ctx.trace_rays(p, o, d)
    assert bad_a == bad_b == 0
    assert (ra.view(np.uint32) == rb.view(np.uint32)).all(), "trace_rays"
    assert counters(sta) == counters(stb)
    ia = {k: v.copy() for k, v in gpu_ctx.intersect_rays(p, o, d)[0].items()}
    ib = ref_ctx.intersect_rays(p, o, d)[0]
    for k in HIT_NAMES:
        assert (ia[k].view(np.uint32) == ib[k].view(np.uint32)).all(), f"intersect_rays {k}"
    assert gpu_ctx.balance_columns(p, 3) == ref_ctx.balance_columns(p, 3)
    h1, _ = gpu_ctx.hit_buffers(p)
    h1 = {k: h1[k].copy() for k in HIT_NAMES}
    h2, _ = ref_ctx.hit_buffers(p)
    for k in HIT_NAMES:
        assert (h1[k].view(np.uint32) == h2[k].view(np.uint32)).all(), f"hit {k}"
    for x, y in zip(gpu_ctx.pick(p, xs, zs), ref_ctx.pick(p, xs, zs)):
        assert (np.asarray(x).view(np.uint32) == np.asarray(y).view(np.uint32)).all(), "pick"
    la = gpu_ctx.occluded_lights(pts)[0].copy()
    assert (la == ref_ctx.occluded_lights(pts)[0]).all(), "occluded_lights"
    want, _, _ = oracle_lights(occ_lib, m, pts)
    assert (la == want).all(), "occluded_lights vs oracle"
    assert (gpu_ctx.occluded_rays(o, d, t)[0] == ref_ctx.occluded_rays(o, d, t)[0]).all(), "occluded_rays"


@gpu
@pytest.mark.parametrize("name", ["sb1_fm1", "sb1_fm2", "grid_fm0"])
def test_interleaved_with_sphere_updates_and_edits(gpu_ctx, ref_ctx, name):
    rec, cam = build(name)
    flat, c = rec.scene.flatten(), cam.export()
    rng = np.random.default_rng(21)
    p = api.default_params(40, 32, 8)
    g = inward_jitter(geom_of(flat), rng, .02, fixed=light_spheres(flat))
    mv = Move.of(variant_moves(name, rec, flat, rng)[0][1])
    e = random_edit(flat, rng)
    want = e.flat(moved_flat(mv.flat(flat), g))
    orders = (("planes", "spheres", "edit"), ("spheres", "planes", "edit"), ("edit", "planes", "spheres"),
              ("edit", "spheres", "planes"))
    for order in orders:
        gpu_ctx.upload_flat(flat, c)
        for step in order:
            if step == "planes":
                mv.apply(gpu_ctx)
            elif step == "spheres":
                gpu_ctx.update_spheres(g)
            else:
                e.apply(gpu_ctx)
        frame_pair(gpu_ctx, ref_ctx, want, c, p, f"{name} {' then '.join(order)}", oracle=order == orders[0])


@gpu
@pytest.mark.parametrize("name", ["sb0_fm2", "sb0_fm3", "sb0_fm0"])
def test_non_finite_and_degenerate_rows(gpu_ctx, ref_ctx, name):
    """Rows the upload takes unchecked: a NaN normal, an infinite origin, a plane of zero extent.  They render as an upload
    of the same rows renders them."""
    rec, cam = build(name)
    flat, c = rec.scene.flatten(), cam.export()
    planes = plane_objects(rec)
    geom, normals, origin = api.plane_rows(flat, planes[:3])
    geom[0, 1] = F32(np.nan)
    normals[0, 1] = F32(np.nan)
    if VARIANTS[name][0] != "infinite":
        geom[1, 7] = geom[1, 11] = F32(0)       # zero extent
        geom[2, 12] = F32(np.inf)
    else:
        geom[1, :3] = F32(0)                    # zero normal
        geom[2, 3] = F32(-np.inf)
    mv = Move(planes[:3], geom, normals, origin)
    gpu_ctx.upload_flat(flat, c)
    mv.apply(gpu_ctx)
    m = mv.flat(flat)
    img, st = gpu_ctx.render(api.default_params(32, 24, 8))
    img = img.copy()
    want, wst = fresh(ref_ctx, m, c).render(api.default_params(32, 24, 8))
    assert (bits(img) == bits(want)).all(), name
    assert counters(st) == counters(wst) or _class(gpu_ctx) != _class(ref_ctx)


@gpu
def test_ordering_and_the_upload_cache(gpu_ctx, ref_ctx):
    rec, cam = build("sb1_fm1")
    flat, c = rec.scene.flatten(), cam.export()
    mv = Move.of(variant_moves("sb1_fm1", rec, flat, np.random.default_rng(2))[0][1])
    flat_b = mv.flat(flat)
    p = api.default_params(64, 48, 6)
    want_a = fresh(ref_ctx, flat, c).render(p)[0].copy()
    want_b = fresh(ref_ctx, flat_b, c).render(p)[0].copy()
    assert not np.array_equal(bits(want_a), bits(want_b))
    bufs = [api.HostBuffer(64 * 48 * 12) for _ in range(3)]
    outs = [b.array(F32, (64, 48, 3)) for b in bufs]
    gpu_ctx.upload_flat(flat, c)
    t1 = gpu_ctx.render_async(p, out=outs[0])
    t2 = gpu_ctx.render_async(p, out=outs[1])
    mv.apply(gpu_ctx)
    gpu_ctx.wait(t1)
    t3 = gpu_ctx.render_async(p, out=outs[2])
    gpu_ctx.wait(t2)
    gpu_ctx.wait(t3)
    assert_bit_identical(outs[0], want_a, "frame 1")
    assert_bit_identical(outs[1], want_a, "frame 2")
    assert_bit_identical(outs[2], want_b, "frame 3")
    gpu_ctx.upload_flat(flat, c)
    mv.apply(gpu_ctx)
    gpu_ctx.upload_flat(flat, c)
    assert gpu_ctx.scene_structures()["clusters"] > 0
    assert_bit_identical(gpu_ctx.render(p)[0], want_a, "upload of the original after an update")


@gpu
@pytest.mark.parametrize("name", ["sb0_fm1", "sb1_fm2"])
def test_errors(gpu_ctx, ref_ctx, name):
    rec, cam = build(name)
    flat, c = rec.scene.flatten(), cam.export()
    n = flat.n_objects
    planes = plane_objects(rec)
    p = api.default_params(32, 24, 6)
    gpu_ctx.upload_flat(flat, c)
    before = gpu_ctx.render(p)[0].copy()
    good = Move.of({o: rigid(rec.calls[o], shift=(.2, .1, 0)) for o in planes[:2]})
    lib = gpu_ctx._lib

    def refused(objs):
        objs = np.asarray(objs, np.int32)
        k = len(objs)
        g, nr, og = (np.resize(a, (k, a.shape[1])).astype(F32) for a in (good.geom, good.normals, good.origin))
        with pytest.raises(api.TcrtError) as e:
            gpu_ctx.update_planes(objs, g, nr, og)
        assert e.value.code == _ffi.TCRT_ERR_INVALID
        assert_bit_identical(gpu_ctx.render(p)[0], before, f"after refusing {objs.tolist()}")

    refused([planes[0], n])
    refused([planes[0], -1])
    refused([planes[0], 0])               # a sphere
    refused([planes[0], planes[1], planes[0]])
    g, nr, og = good.geom, good.normals, good.origin
    objs = good.objects
    for rc in (lib.tcrt_update_planes(gpu_ctx._h, -1, objs.ctypes.data, g.ctypes.data, nr.ctypes.data, og.ctypes.data, None),
               lib.tcrt_update_planes(gpu_ctx._h, 2, None, g.ctypes.data, nr.ctypes.data, og.ctypes.data, None),
               lib.tcrt_update_planes(gpu_ctx._h, 2, objs.ctypes.data, None, nr.ctypes.data, og.ctypes.data, None),
               lib.tcrt_update_planes(gpu_ctx._h, 2, objs.ctypes.data, g.ctypes.data, None, og.ctypes.data, None),
               lib.tcrt_update_planes(gpu_ctx._h, 2, objs.ctypes.data, g.ctypes.data, nr.ctypes.data, None, None)):
        assert rc == _ffi.TCRT_ERR_INVALID
    assert_bit_identical(gpu_ctx.render(p)[0], before, "after n < 0 and NULL arrays")
    st = gpu_ctx.update_planes(np.zeros(0, np.int32), np.zeros((0, 16), F32), np.zeros((0, 8), F32),
                               np.zeros((0, 4), F32))
    assert st.gpu_launches == 0
    good.apply(gpu_ctx)
    frame_pair(gpu_ctx, ref_ctx, good.flat(flat), c, p, f"{name} valid update after refused ones", oracle=True)
    new = api.Context([0])
    try:
        with pytest.raises(api.TcrtError) as e:
            good.apply(new)
        assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
    finally:
        new.close()


@gpu
@pytest.mark.parametrize("second", ["same device", "second device"])
def test_two_slots(gpu_ctx, second):
    if second == "second device" and api.device_count() < 2:
        pytest.skip("one GPU visible")
    rec, cam = build("sb1_fm1")
    flat, c = rec.scene.flatten(), cam.export()
    steps = variant_moves("sb1_fm1", rec, flat, np.random.default_rng(5))
    p = api.default_params(64, 48, 8)
    gpu_ctx.upload_flat(flat, c)
    for _, calls, _ in steps:
        Move.of(calls).apply(gpu_ctx)
    want, st = gpu_ctx.render(p)
    want = want.copy()
    pair = api.Context([0, 0 if second == "same device" else 1])
    try:
        pair.upload_flat(flat, c)
        for _, calls, _ in steps:
            st2 = Move.of(calls).apply(pair)
            assert st2.n_devices == 2
        img, st3 = pair.render(p)
        assert_bit_identical(img, want, f"two slots ({second})")
        assert counters(st3) == counters(st)
    finally:
        pair.close()


CPP_PROGRAM = r"""
#include <stdio.h>
#include <vector>
#include "Camera.h"
#include "RayTracer.h"
#include "Scene.h"

using namespace CelioRayTracer;

// a room, a floor and a few spheres; `moved`: the room shifted and the floor tilted, in the same object order
static void build(Scene& s, bool moved) {
    for (int i = 0; i < 4; i++) s.addObject(new SceneSphere(vector3d(-1.5f + i, 1.0f + .5f * i, 1.5f), .6f));
    SceneSphere* light = new SceneSphere(vector3d(1.0f, 3.0f, 5.0f), .2f);
    light->setAsLightSource();
    s.addObject(light);
    s.addObject(new SceneInfinitePlane(vector3d(0, 0, -.5f), moved ? vector3d(.05f, .1f, 1) : vector3d(0, 0, 1),
                                       vector3d(1, 0, 0)));
    SceneFinitePlane** box = s.makeSceneBox(moved ? vector3d(-6.5f, -5.75f, -1) : vector3d(-6, -6, -1), vector3d(12, 14, 9));
    for (int k = 0; k < 6; k++) s.addObject(box[k]);   // makeSceneBox only builds the faces
}

int main() {
    Scene scene, moved, other;
    Camera camera;
    build(scene, false);
    build(moved, true);
    other.initialize();
    const int W = 48, H = 40;
    GpuRayTracer rt;
    RenderSettings rs;
    rs.width = W; rs.height = H; rs.max_depth = 8;
    std::vector<float> rgb(W * H * 3);
    if (!rt.ok() || rt.setScene(scene, camera)) return 1;
    const int objs[7] = {5, 6, 7, 8, 9, 10, 11};
    if (rt.updatePlanes(moved, objs, 7) || rt.render(rs, rgb.data())) {
        fprintf(stderr, "%s\n", rt.lastError());
        return 1;
    }
    const int sphere[1] = {0};
    printf("%d %d\n", rt.updatePlanes(moved, sphere, 1), rt.updatePlanes(other, objs, 7));   // both refused
    FILE* f = fopen("moved.bin", "wb");
    if (!f) return 1;
    fwrite(rgb.data(), 4, rgb.size(), f);
    return fclose(f) ? 1 : 0;
}
"""


def cpp_scene(moved):
    s = api.Scene()
    for i in range(4):
        s.addSphere((-1.5 + i, 1.0 + .5 * i, 1.5), .6)
    s.addSphere((1.0, 3.0, 5.0), .2).setAsLightSource()
    s.addInfinitePlane((0, 0, -.5), (.05, .1, 1) if moved else (0, 0, 1), (1, 0, 0))
    s.makeSceneBox((-6.5, -5.75, -1) if moved else (-6, -6, -1), (12, 14, 9))
    return s


@gpu
def test_cpp_update_planes(gpu_ctx, tmp_path):
    src = tmp_path / "move.cpp"
    src.write_text(CPP_PROGRAM)
    libdir = os.path.join(ROOT, "tilecoderaytracer_b200")
    exe = tmp_path / "move"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), str(src),
                    "-L", libdir, "-ltcrt", f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert [int(x) for x in r.stdout.split()[-2:]] == [_ffi.TCRT_ERR_INVALID] * 2
    got = np.frombuffer((tmp_path / "moved.bin").read_bytes(), F32).reshape(48, 40, 3)
    scene, cam = cpp_scene(True), api.Camera()
    gpu_ctx.upload(scene, cam)
    p = api.default_params(48, 40, 8)
    want, _ = gpu_ctx.render(p)
    assert_bit_identical(got, want, "C++ updatePlanes")
    o, _ = O.render(scene.flatten(), cam.export(), p)
    assert_bit_identical(got, o, "C++ updatePlanes vs oracle")
