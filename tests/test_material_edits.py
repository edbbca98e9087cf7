"""Material edits (tcrt_update_materials, tcrt_update_textures): new colours, shading factors, light intensities, texture
ids and checker rows for the resident scene, written on the GPU in place.  After an edit every call that reads the scene
must return, bit for bit, what it returns after a fresh tcrt_upload_scene of the edited scene, and for small frames what
the oracle renders of it; NaN where the reference makes NaN, which needs the dead-path bound to follow the edits."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import assert_bit_identical, bits, make_scene
from test_dead_paths import assert_same_bits_or_both_nan, dying_scene
from test_kernel_variants import NAMES, build
from test_occlusion import occ_lib, oracle_lights  # noqa: F401  (occ_lib is a fixture)
from test_scene_updates import _class, counters, frame_pair, fresh, geom_of, light_spheres, moved_flat, ref_ctx  # noqa: F401

gpu = pytest.mark.gpu
F32 = np.float32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENTRY_POINTS = ("tcrt_update_materials", "tcrt_update_textures")
HIT_NAMES = ("object", "distance", "normal")


# ---- edited copies of flattened scenes -----------------------------------------------------------------------------------

def _rows(flat, name, width, count, dtype=F32):
    if count == 0:
        return np.zeros((0, width), dtype)
    return np.ctypeslib.as_array(getattr(flat, name), (count * width,)).reshape(count, width).astype(dtype)


def texture_rows(flat):
    return _rows(flat, "textures", 8, flat.n_textures)


class Edit:
    """Rows for update_materials (objects, surface, material, texture; any part None) and update_textures (ids, rows)."""

    def __init__(self, objects=(), surface=None, material=None, texture=None, tex_ids=(), tex_rows=None):
        self.objects = np.asarray(objects, np.int32)
        self.surface, self.material, self.texture = surface, material, texture
        self.tex_ids = np.asarray(tex_ids, np.int32)
        self.tex_rows = tex_rows

    def apply(self, ctx):
        """Both calls; the stats of the object rows (of the checker rows when there are none)."""
        st = None
        if len(self.objects):
            st = ctx.update_materials(self.objects, self.surface, self.material, self.texture)
        if len(self.tex_ids):
            st2 = ctx.update_textures(self.tex_ids, self.tex_rows)
            st = st or st2
        return st

    def flat(self, flat):
        """A copy of the flattened scene with these rows replaced: the scene an edit must be indistinguishable from."""
        m = _ffi.TcrtScene.from_buffer_copy(bytes(flat))
        n = flat.n_objects
        surface = _rows(flat, "obj_surface", 4, n).copy()
        material = _rows(flat, "obj_material", 4, n).copy()
        info = _rows(flat, "obj_info", 4, n, np.int32).copy()
        tex = texture_rows(flat).copy()
        if self.surface is not None:
            surface[self.objects] = self.surface
        if self.material is not None:
            material[self.objects, :3] = self.material[:, :3]
        if self.texture is not None:
            info[self.objects, 3] = self.texture
        if len(self.tex_ids):
            tex[self.tex_ids] = self.tex_rows
        m.obj_surface = surface.ctypes.data_as(_ffi.c_float_p)
        m.obj_material = material.ctypes.data_as(_ffi.c_float_p)
        m.obj_info = info.ctypes.data_as(_ffi.c_int_p)
        m.textures = tex.ctypes.data_as(_ffi.c_float_p) if len(tex) else None
        m._keep = (surface, material, info, tex, flat)
        return m


def whole_scene_edit(target):
    """Every object's rows and every checker row of `target`."""
    objs = np.arange(target.n_objects, dtype=np.int32)
    s, m, t = api.material_rows(target, objs)
    return Edit(objs, s, m, t, np.arange(target.n_textures), texture_rows(target))


def random_edit(flat, rng, frac=1 / 3):
    """A third of the objects: new colours, diffuse and specular factors, reflective 0 <-> 1 (or a new value), lights'
    colours and intensities, texture ids reassigned; and every checker row new."""
    n, n_tex = flat.n_objects, flat.n_textures
    objs = np.sort(rng.choice(n, max(1, int(n * frac)), replace=False)).astype(np.int32)
    s, m, t = api.material_rows(flat, objs)
    s[:, :3] = rng.uniform(0, 1, (len(objs), 3)).astype(F32)
    s[:, 3] = rng.uniform(0, 1, len(objs)).astype(F32)
    m[:, 0] = rng.uniform(0, 1, len(objs)).astype(F32)
    m[:, 1] = np.where(m[:, 1] > 0, F32(0), F32(1))
    m[::4, 1] = rng.uniform(.2, .8, len(m[::4])).astype(F32)
    info = _rows(flat, "obj_info", 4, n, np.int32)
    lights = info[objs, 2] != 0
    m[lights, 2] = rng.uniform(.5, 3, int(lights.sum())).astype(F32)
    m[:, 3] = F32(7)          # ignored
    t = rng.integers(-1, n_tex, len(objs)).astype(np.int32) if n_tex else t
    rows = texture_rows(flat).copy()
    if n_tex:
        rows[:, [0, 1, 2, 4, 5, 6]] = rng.uniform(0, 1, (n_tex, 6)).astype(F32)
        rows[:, [3, 7]] *= F32(1.5)
    return Edit(objs, s, m, t, np.arange(n_tex), rows)


# ---- without a GPU ---------------------------------------------------------------------------------------------------------

def test_entry_points_are_exported():
    lib = _ffi.load()
    for name in ENTRY_POINTS:
        assert hasattr(lib, name), name


def test_entry_points_refuse_a_null_context():
    lib = _ffi.load()
    objs = np.zeros(1, np.int32)
    rows = np.zeros((1, 8), F32)
    p, r = objs.ctypes.data_as(C.c_void_p), rows.ctypes.data_as(C.c_void_p)
    assert lib.tcrt_update_materials(None, 1, p, r, r, p, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_update_textures(None, 1, p, r, None) == _ffi.TCRT_ERR_INVALID


def test_material_rows_are_the_flattened_scene():
    s = api.Scene()
    refs = [s.addSphere((k, 0, 0), .5) for k in range(6)]
    s.addInfinitePlane((0, 0, -1), (0, 0, 1), (1, 0, 0)).setCheckerBoard((1, .5, .25), (0, .1, .2), 1.5, 2.5)
    refs[0].setColor(.1, .2, .3)
    refs[1].setDiffuseFactor(1 / 3)
    refs[2].setSpecularFactor(.7)
    refs[3].setReflectiveFactor(.9)
    refs[4].setAsLightSource(2.5).setColor(1e-12, float("nan"), -0.0)
    objs = [6, 4, 0, 1, 2, 3]
    flat = s.flatten()
    surface, material, texture = api.material_rows(flat, objs)
    assert surface.dtype == F32 and material.dtype == F32 and texture.dtype == np.int32
    assert surface.shape == (6, 4) and material.shape == (6, 4) and texture.shape == (6,)
    assert (bits(surface) == bits(_rows(flat, "obj_surface", 4, 7)[objs])).all()
    assert (bits(material) == bits(_rows(flat, "obj_material", 4, 7)[objs])).all()
    assert texture.tolist() == [0, -1, -1, -1, -1, -1]
    # the setters' values, as binary32 bit patterns
    assert (bits(surface[1, :3]) == bits(np.array([1e-12, np.nan, -0.0], F32))).all()
    assert bits(material[1, 2]) == bits(F32(2.5))
    assert (bits(surface[2, :3]) == bits(np.array([.1, .2, .3], F32))).all()
    assert bits(surface[3, 3]) == bits(F32(1 / 3))
    assert bits(material[4, 0]) == bits(F32(.7))
    assert bits(material[5, 1]) == bits(F32(.9))


def test_edited_flat_is_a_fresh_build():
    """Edit.flat of a flattened scene is what the host API builds from the edited scene."""
    def scene(edited):
        s = api.Scene()
        floor = s.addInfinitePlane((0, 0, -4), (0, 0, 1), (1, 0, 0)).setCheckerBoard((1, 1, 1), (0, 0, 0), 2, 2)
        a = s.addSphere((0, 0, 0), 1).setColor(.5, .5, .5).setReflectiveFactor(1)
        light = s.addSphere((3, 3, 3), .2).setAsLightSource(1.0)
        if edited:
            a.setColor(.25, 0, 1).setReflectiveFactor(0).setDiffuseFactor(.4).setSpecularFactor(.1)
            light.setColor(.9, .8, .7).setAsLightSource(3.0)
            floor.setCheckerBoard((.5, .5, 1), (.1, 0, 0), 3, 1)   # a new checker object: flattened in the same slot
        return s

    s0, s1 = scene(False), scene(True)           # the flattened scenes point into them
    f0, f1 = s0.flatten(), s1.flatten()
    objs = [1, 2]
    e = Edit(objs, *api.material_rows(f1, objs), tex_ids=[0], tex_rows=texture_rows(f1))
    m = e.flat(f0)
    for name, width, count in (("obj_surface", 4, 3), ("obj_material", 4, 3), ("obj_info", 4, 3), ("textures", 8, 1)):
        a = np.ctypeslib.as_array(getattr(m, name), (width * count,))
        b = np.ctypeslib.as_array(getattr(f1, name), (width * count,))
        assert (a.view(np.uint32) == b.view(np.uint32)).all(), name


# ---- on the GPU ------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("depth", [0, 8, 64])
@pytest.mark.parametrize("name", NAMES)
def test_every_dispatch_class(gpu_ctx, ref_ctx, name, depth):
    s, cam = build(name)
    flat, c = s.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    cls = _class(gpu_ctx)
    rng = np.random.default_rng(100 + depth + len(name))
    e = random_edit(flat, rng)
    st = e.apply(gpu_ctx)
    assert counters(st) == (0, 0, 0) and st.gpu_launches == 1
    assert _class(gpu_ctx) == cls, f"{name}: the edit changed the dispatch class"
    p = api.default_params(32, 24, depth)
    frame_pair(gpu_ctx, ref_ctx, e.flat(flat), c, p, f"{name} d{depth}", oracle=depth <= 8)


def _dead_pair(ctx, ref, flat, c, p, what, prunes, nan=None):
    """The edited context against a fresh upload of `flat` and the oracle: the same bits or NaN on both sides, the same
    counters; the dead-path decision of the scene, and whether the oracle's frame has NaN (None: either)."""
    assert api.plan_dead_paths(flat, p) == prunes, what
    img, st = ctx.render(p)
    img = img.copy()
    want, wst = fresh(ref, flat, c).render(p)
    assert_same_bits_or_both_nan(img, want, f"{what} vs fresh upload")
    assert counters(st) == counters(wst), what
    o, cnt = O.render(flat, c, p)
    assert_same_bits_or_both_nan(img, o, f"{what} vs oracle")
    assert counters(st) == (cnt["rays_primary"], cnt["rays_shadow"], cnt["rays_reflect"]), what
    if nan is not None:
        assert np.isnan(o).any() == nan, what


@gpu
@pytest.mark.parametrize("kind", ["grid", "planes"])
def test_dead_paths_follow_the_edits(gpu_ctx, ref_ctx, kind):
    """primary -> tiny_colours -> primary by edits alone: the second overflows and makes NaN in the reference, so the
    grid kernel must stop pruning, and prune again after the edit back."""
    cam = api.Camera()
    c = cam.export()
    prim_s, tiny_s = dying_scene("primary", kind), dying_scene("tiny_colours", kind)
    prim, tiny = prim_s.flatten(), tiny_s.flatten()
    assert prim.n_objects == tiny.n_objects and prim.n_textures == tiny.n_textures == 1
    p = api.default_params(96, 64, 8)
    gpu_ctx.upload_flat(prim, c)
    assert (gpu_ctx.scene_structures()["grid_cells"] > 0) == (kind == "grid")
    for target, prunes, what in ((tiny, False, "tiny_colours"), (prim, True, "primary again")):
        whole_scene_edit(target).apply(gpu_ctx)
        _dead_pair(gpu_ctx, ref_ctx, target, c, p, f"{kind} {what}", prunes, nan=not prunes)


@gpu
@pytest.mark.parametrize("kind", ["grid", "planes"])
def test_dead_paths_overflow_nan_and_negative_zero(gpu_ctx, ref_ctx, kind):
    c = api.Camera().export()
    prim_s = dying_scene("primary", kind)        # the flattened scene points into it
    prim = prim_s.flatten()
    p = api.default_params(96, 64, 10)
    n = prim.n_objects
    info = _rows(prim, "obj_info", 4, n, np.int32)
    mirrors = np.array([i for i in range(n) if not info[i, 2] and info[i, 0] != 2], np.int32)   # no lights, no floor
    light = int(np.nonzero(info[:, 2])[0][0])
    gpu_ctx.upload_flat(prim, c)
    # one light at 3e38, the mirrors' colours doubled: a mirror's child overflows to inf, a zero channel makes NaN
    s, m, t = api.material_rows(prim, np.r_[light, mirrors])
    m[0, 2] = F32(3e38)
    s[1:, :3] *= F32(2)
    e = Edit(np.r_[light, mirrors], s, m, t)
    e.apply(gpu_ctx)
    over = e.flat(prim)
    assert not api.plan_dead_paths(over, p)
    img, st = gpu_ctx.render(p)
    img = img.copy()
    want, wst = fresh(ref_ctx, over, c).render(p)
    assert_same_bits_or_both_nan(img, want, f"{kind} 3e38 vs fresh upload")
    assert counters(st) == counters(wst)
    o, cnt = O.render(over, c, p)
    assert_same_bits_or_both_nan(img, o, f"{kind} 3e38 vs oracle")
    assert counters(st) == (cnt["rays_primary"], cnt["rays_shadow"], cnt["rays_reflect"])
    # back to the primary materials: pruning on again
    whole_scene_edit(prim).apply(gpu_ctx)
    _dead_pair(gpu_ctx, ref_ctx, prim, c, p, f"{kind} primary after 3e38", True)
    # a NaN colour: pruning off; NaN colours render as the reference renders them
    s, m, t = api.material_rows(prim, mirrors[:1])
    s[0, 1] = F32(np.nan)
    e = Edit(mirrors[:1], surface=s)
    e.apply(gpu_ctx)
    _dead_pair(gpu_ctx, ref_ctx, e.flat(prim), c, p, f"{kind} nan colour", False)
    # -0 instead of every zero colour channel (and the NaN gone): pruning on
    s, m, t = api.material_rows(prim, mirrors)
    s[:, :3] = np.where(s[:, :3] == 0, F32(-0.0), s[:, :3])
    e = Edit(mirrors, surface=s)
    e.apply(gpu_ctx)
    _dead_pair(gpu_ctx, ref_ctx, e.flat(prim), c, p, f"{kind} negative zero", True)


@gpu
@pytest.mark.parametrize("name", ["sb1_fm1", "grid_fm0"])
def test_every_other_reader(gpu_ctx, ref_ctx, occ_lib, name):
    from test_views import three_views

    s, cam = build(name)
    flat, c = s.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    rng = np.random.default_rng(4)
    p = api.default_params(40, 32, 8)
    xs, zs = rng.integers(0, 40, 30), rng.integers(0, 32, 30)
    g = geom_of(flat)
    pts = np.concatenate([g[:, :3] + F32(.5), rng.uniform(-6, 6, (500, 3)).astype(F32)]).astype(F32)
    o = np.array(c.eye[:], F32)
    d = api.normalize_like_reference(rng.normal(0, 1, (400, 3)).astype(F32))
    t = rng.uniform(.5, 20, 400).astype(F32)

    def hits_and_shadows(ctx):
        h, _ = ctx.hit_buffers(p)
        out = {k: h[k].copy() for k in HIT_NAMES}
        out["pick"] = [x.copy() for x in ctx.pick(p, xs, zs)]
        out["lights"] = ctx.occluded_lights(pts)[0].copy()
        out["rays"] = ctx.occluded_rays(o, d, t)[0].copy()
        return out

    def same(a, b, what):
        for k in HIT_NAMES:
            assert (a[k].view(np.uint32) == b[k].view(np.uint32)).all(), f"{what} {k}"
        for x, y in zip(a["pick"], b["pick"]):
            assert (x.view(np.uint32) == y.view(np.uint32)).all(), f"{what} pick"
        assert (a["lights"] == b["lights"]).all(), f"{what} occluded_lights"
        assert (a["rays"] == b["rays"]).all(), f"{what} occluded_rays"

    before = hits_and_shadows(gpu_ctx)
    e = random_edit(flat, rng)
    e.apply(gpu_ctx)
    m = e.flat(flat)
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
    assert gpu_ctx.balance_columns(p, 3) == ref_ctx.balance_columns(p, 3)
    after = hits_and_shadows(gpu_ctx)
    same(after, before, "unchanged by the edit")
    same(after, hits_and_shadows(ref_ctx), "vs fresh upload")
    want, _, _ = oracle_lights(occ_lib, m, pts)
    assert (after["lights"] == want).all(), "occluded_lights vs oracle"


def _light_edit(flat, rng):
    """Every light: a new colour and intensity."""
    n = flat.n_objects
    info = _rows(flat, "obj_info", 4, n, np.int32)
    lights = np.nonzero(info[:, 2])[0].astype(np.int32)
    s, m, t = api.material_rows(flat, lights)
    s[:, :3] = rng.uniform(.3, 1, (len(lights), 3)).astype(F32)
    m[:, 2] = rng.uniform(.5, 4, len(lights)).astype(F32)
    return Edit(lights, s, m)


@gpu
@pytest.mark.parametrize("name", ["sb1_fm1", "grid_fm0"])
def test_edits_and_sphere_updates_interleaved(gpu_ctx, ref_ctx, name):
    """A sphere update rewrites every light row from the host's copy of the lights: an edit made before it must stay,
    and one made after it must leave the moved positions (and the room's inside masks) in place."""
    s, cam = build(name)
    flat, c = s.flatten(), cam.export()
    rng = np.random.default_rng(9)
    p = api.default_params(48, 32, 8)
    g0 = geom_of(flat)
    g = g0.copy()
    g[:, :3] += rng.normal(0, .02, (len(g), 3)).astype(F32)
    lights = light_spheres(flat)
    g[lights[0], :3] += np.array([.3, -.2, .1], F32)
    e = _light_edit(flat, rng)
    # edit, then move
    gpu_ctx.upload_flat(flat, c)
    e.apply(gpu_ctx)
    gpu_ctx.update_spheres(g)
    want = e.flat(moved_flat(flat, g))
    frame_pair(gpu_ctx, ref_ctx, want, c, p, f"{name} edit then move", oracle=True)
    # move, then edit
    gpu_ctx.upload_flat(flat, c)
    gpu_ctx.update_spheres(g)
    e.apply(gpu_ctx)
    frame_pair(gpu_ctx, ref_ctx, want, c, p, f"{name} move then edit", oracle=True)
    # and once more both ways round on the same context
    e2 = _light_edit(flat, rng)
    e2.apply(gpu_ctx)
    gpu_ctx.update_spheres(g0)
    frame_pair(gpu_ctx, ref_ctx, e2.flat(flat), c, p, f"{name} second edit, moved back")


@gpu
def test_ordering_and_the_upload_cache(gpu_ctx, ref_ctx):
    scene, cam = make_scene("synth256")
    flat, c = scene.flatten(), cam.export()
    e = random_edit(flat, np.random.default_rng(12))
    flat_b = e.flat(flat)
    p = api.default_params(64, 48, 6)
    want_a, _ = fresh(ref_ctx, flat, c).render(p)
    want_a = want_a.copy()
    want_b, _ = fresh(ref_ctx, flat_b, c).render(p)
    want_b = want_b.copy()
    assert not np.array_equal(bits(want_a), bits(want_b))
    bufs = [api.HostBuffer(64 * 48 * 12) for _ in range(3)]
    outs = [b.array(F32, (64, 48, 3)) for b in bufs]
    gpu_ctx.upload_flat(flat, c)
    t1 = gpu_ctx.render_async(p, out=outs[0])
    t2 = gpu_ctx.render_async(p, out=outs[1])
    e.apply(gpu_ctx)
    gpu_ctx.wait(t1)
    t3 = gpu_ctx.render_async(p, out=outs[2])
    gpu_ctx.wait(t2)
    gpu_ctx.wait(t3)
    assert_bit_identical(outs[0], want_a, "frame 1")
    assert_bit_identical(outs[1], want_a, "frame 2")
    assert_bit_identical(outs[2], want_b, "frame 3")
    # an edit makes the next upload rebuild: the original scene again is the original scene
    gpu_ctx.upload_flat(flat, c)
    e.apply(gpu_ctx)
    gpu_ctx.upload_flat(flat, c)
    assert_bit_identical(gpu_ctx.render(p)[0], want_a, "upload of the original after an edit")
    e.apply(gpu_ctx)
    gpu_ctx.upload_flat(flat_b, c)
    assert_bit_identical(gpu_ctx.render(p)[0], want_b, "upload of the edited scene after the edit")


@gpu
@pytest.mark.parametrize("name", ["sb0_fm1", "grid_fm0"])
def test_errors(gpu_ctx, ref_ctx, name):
    """Every refused call leaves the frame as it was; a later valid edit, which sends rows the refused calls listed,
    matches its fresh upload, and so does a sphere update, which rewrites the light rows from the host: nothing of a
    refused call reached the host's copy of the materials either."""
    s, cam = build(name)
    flat, c = s.flatten(), cam.export()
    n, n_tex = flat.n_objects, flat.n_textures
    assert n_tex >= 1
    info = _rows(flat, "obj_info", 4, n, np.int32)
    light = int(np.nonzero(info[:, 2])[0][0])
    p = api.default_params(32, 24, 6)
    gpu_ctx.upload_flat(flat, c)
    before = gpu_ctx.render(p)[0].copy()
    objs = np.array([light, 3], np.int32)
    s_bad, m_bad, t_ok = api.material_rows(flat, objs)
    s_bad[:, :3] = F32(.123)
    m_bad[:, 2] = F32(9)
    tex_rows = texture_rows(flat) * F32(.5)
    lib = gpu_ctx._lib

    def refused(fn, *args):
        with pytest.raises(api.TcrtError) as e:
            fn(*args)
        assert e.value.code == _ffi.TCRT_ERR_INVALID
        assert_bit_identical(gpu_ctx.render(p)[0], before, f"after {fn.__name__}{args[:1]}")

    for bad in (n, -1):
        o = np.r_[objs, bad].astype(np.int32)
        refused(gpu_ctx.update_materials, o, np.r_[s_bad, s_bad[:1]], np.r_[m_bad, m_bad[:1]], np.r_[t_ok, -1])
    refused(gpu_ctx.update_materials, np.r_[objs, objs[0]], np.r_[s_bad, s_bad[:1]], None, None)       # duplicate
    for tid in (n_tex, -2):
        refused(gpu_ctx.update_materials, objs, s_bad, m_bad, np.array([t_ok[0], tid], np.int32))
    refused(gpu_ctx.update_materials, objs)                                                             # all NULL
    for bad in (n_tex, -1):
        refused(gpu_ctx.update_textures, np.array([0, bad], np.int32), np.r_[tex_rows[:1], tex_rows[:1]])
    refused(gpu_ctx.update_textures, np.array([0, 0], np.int32), np.r_[tex_rows[:1], tex_rows[:1]])      # duplicate
    # n < 0 and NULL arrays with n > 0, through the C entry points
    for rc in (lib.tcrt_update_materials(gpu_ctx._h, -1, objs.ctypes.data, s_bad.ctypes.data, None, None, None),
               lib.tcrt_update_materials(gpu_ctx._h, 2, None, s_bad.ctypes.data, None, None, None),
               lib.tcrt_update_textures(gpu_ctx._h, -1, objs.ctypes.data, tex_rows.ctypes.data, None),
               lib.tcrt_update_textures(gpu_ctx._h, 1, None, tex_rows.ctypes.data, None),
               lib.tcrt_update_textures(gpu_ctx._h, 1, objs.ctypes.data, None, None)):
        assert rc == _ffi.TCRT_ERR_INVALID
    assert_bit_identical(gpu_ctx.render(p)[0], before, "after n < 0 and NULL arrays")
    # a valid edit of the same objects that sends only the specular factors: the colours and intensities come from the
    # host's copy, which must still hold the uploaded ones
    _, m_ok, _ = api.material_rows(flat, objs)
    m_ok[:, 0] = F32(.25)
    e = Edit(objs, material=m_ok)
    st = e.apply(gpu_ctx)
    assert st.gpu_launches == 1
    frame_pair(gpu_ctx, ref_ctx, e.flat(flat), c, p, f"{name} valid edit after refused ones", oracle=True)
    gpu_ctx.update_spheres(geom_of(flat))
    frame_pair(gpu_ctx, ref_ctx, e.flat(flat), c, p, f"{name} sphere update after refused edits")
    st = gpu_ctx.update_materials(np.zeros(0, np.int32), np.zeros((0, 4), F32))
    assert st.gpu_launches == 0
    st = gpu_ctx.update_textures(np.zeros(0, np.int32), np.zeros((0, 8), F32))
    assert st.gpu_launches == 0
    new = api.Context([0])
    try:
        with pytest.raises(api.TcrtError) as e:
            new.update_materials(objs, s_bad)
        assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
        with pytest.raises(api.TcrtError) as e:
            new.update_textures([0], tex_rows[:1])
        assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
    finally:
        new.close()


@gpu
@pytest.mark.parametrize("second", ["same device", "second device"])
def test_two_slots(gpu_ctx, second):
    n_dev = api.device_count()
    if second == "second device" and n_dev < 2:
        pytest.skip("one GPU visible")
    s, cam = make_scene("synth256")
    flat, c = s.flatten(), cam.export()
    e = random_edit(flat, np.random.default_rng(5))
    p = api.default_params(64, 48, 8)
    gpu_ctx.upload_flat(flat, c)
    e.apply(gpu_ctx)
    want, st = gpu_ctx.render(p)
    want = want.copy()
    pair = api.Context([0, 0 if second == "same device" else 1])
    try:
        pair.upload_flat(flat, c)
        st2 = e.apply(pair)
        assert st2.n_devices == 2 and st2.gpu_launches == 2
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

int main() {
    using namespace CelioRayTracer;
    Scene scene;
    Camera camera;
    if (scene.initialize()) return 1;
    const int W = 48, H = 40;
    GpuRayTracer rt;
    RenderSettings rs;
    rs.width = W; rs.height = H; rs.max_depth = 50;
    std::vector<float> rgb(W * H * 3);
    if (!rt.ok() || rt.setScene(scene, camera)) return 1;
    const int objs[3] = {3, 5, 8};
    ObjMaterial* m = scene.getObject(3)->getMaterial();
    m->setColor(vector3d(.2f, .9f, .4f));
    m->setReflectiveFactor(0.f);
    scene.getObject(5)->getMaterial()->setDiffuseFactor(.25f);
    scene.getObject(8)->getMaterial()->setSpecularFactor(.125f);
    if (rt.updateMaterials(scene, objs, 3) || rt.render(rs, rgb.data())) {
        fprintf(stderr, "%s\n", rt.lastError());
        return 1;
    }
    scene.getObject(9)->setAsLightSource();   // a new light needs setScene
    printf("%d\n", rt.updateMaterials(scene, objs, 3));
    FILE* f = fopen("edited.bin", "wb");
    if (!f) return 1;
    fwrite(rgb.data(), 4, rgb.size(), f);
    return fclose(f) ? 1 : 0;
}
"""


@gpu
def test_cpp_update_materials(gpu_ctx, tmp_path):
    src = tmp_path / "edit.cpp"
    src.write_text(CPP_PROGRAM)
    libdir = os.path.join(ROOT, "tilecoderaytracer_b200")
    exe = tmp_path / "edit"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), str(src),
                    "-L", libdir, "-ltcrt", f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert int(r.stdout.split()[-1]) == _ffi.TCRT_ERR_INVALID
    got = np.frombuffer((tmp_path / "edited.bin").read_bytes(), F32).reshape(48, 40, 3)
    scene, cam = make_scene("default")
    scene._obj(3).setColor(.2, .9, .4).setReflectiveFactor(0.0)
    scene._obj(5).setDiffuseFactor(.25)
    scene._obj(8).setSpecularFactor(.125)
    gpu_ctx.upload(scene, cam)
    want, _ = gpu_ctx.render(api.default_params(48, 40, 50))
    assert_bit_identical(got, want, "C++ updateMaterials")
    o, _ = O.render(scene.flatten(), cam.export(), api.default_params(48, 40, 50))
    assert_bit_identical(got, o, "C++ updateMaterials vs oracle")
