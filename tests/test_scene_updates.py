"""Moving spheres (tcrt_update_spheres and its device form): new centres and radii for the resident scene's spheres, applied
on the GPU by refitting the sphere BVH and re-registering the sphere grid.  After an update every call that reads the scene
must return, bit for bit, what it returns after a fresh tcrt_upload_scene of the moved scene — the same scene with
sphere_geom replaced and each sphere's obj_origin row (a light sphere's position) at its new centre — and, for small
frames, what the oracle renders of it."""
import ctypes as C

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import assert_bit_identical, make_scene
from test_kernel_variants import NAMES, VARIANTS, ROOM_LO, ROOM_DIMS, build
from test_occlusion import occ_lib, oracle_lights  # noqa: F401  (occ_lib is a fixture)
from test_ray_batches import oracle_hits, oracle_trace, rays_lib  # noqa: F401  (rays_lib is a fixture)

gpu = pytest.mark.gpu
F32 = np.float32
ENTRY_POINTS = ("tcrt_update_spheres", "tcrt_update_spheres_device")
HIT_NAMES = ("object", "distance", "normal")


# ---- scenes and their moved copies ---------------------------------------------------------------------------------------

def geom_of(flat):
    n = flat.n_spheres
    return np.ctypeslib.as_array(flat.sphere_geom, (n * 4,)).reshape(n, 4).astype(F32) if n else np.zeros((0, 4), F32)


def moved_flat(flat, geom):
    """A copy of the flattened scene with sphere_geom = geom and each sphere's obj_origin row at its new centre: the scene
    an update to geom must be indistinguishable from.  The arrays live on the returned struct."""
    m = _ffi.TcrtScene.from_buffer_copy(bytes(flat))
    g = np.ascontiguousarray(geom, F32).copy()
    n_obj = flat.n_objects
    origin = np.ctypeslib.as_array(flat.obj_origin, (n_obj * 4,)).reshape(n_obj, 4).copy()
    objs = np.ctypeslib.as_array(flat.sphere_obj, (flat.n_spheres,)) if flat.n_spheres else np.zeros(0, np.int32)
    for i, o in enumerate(objs):
        origin[o, :3] = g[i, :3]
    m.sphere_geom = g.ctypes.data_as(_ffi.c_float_p)
    m.obj_origin = origin.ctypes.data_as(_ffi.c_float_p)
    m._keep = (g, origin, flat)
    return m


def light_spheres(flat):
    """Indices of the spheres that are lights."""
    n_obj = flat.n_objects
    info = np.ctypeslib.as_array(flat.obj_info, (n_obj * 4,)).reshape(n_obj, 4)
    objs = np.ctypeslib.as_array(flat.sphere_obj, (flat.n_spheres,))
    return [i for i, o in enumerate(objs) if info[o, 2]]


def spacing(geom):
    """Median nearest-neighbour distance of the centres (a lattice's spacing)."""
    c = geom[:, :3].astype(np.float64)
    d = np.sqrt(((c[:, None, :] - c[None, :, :]) ** 2).sum(-1))
    np.fill_diagonal(d, np.inf)
    return float(np.median(d.min(1)))


def inward_jitter(geom, rng, scale, fixed=()):
    """Centres jittered by `scale` (a standard deviation), except that a sphere within half the spacing of the bounding
    box of the moving centres moves only inwards along that axis: every sphere stays inside the box the upload fitted its
    grid to (the grid keeps its origin, cell size and dimensions, and the upload leaves only about 1/50 of a cell between
    the outermost spheres' boxes and the grid's walls).  Spheres in `fixed` (the lights) stay."""
    moving = ~np.isin(np.arange(len(geom)), list(fixed))
    s = spacing(geom[moving])
    lo, hi = geom[moving, :3].min(0), geom[moving, :3].max(0)
    d = rng.normal(0.0, scale, (len(geom), 3)).astype(F32)
    d = np.where(geom[:, :3] < lo + 0.5 * s, np.abs(d), d)
    d = np.where(geom[:, :3] > hi - 0.5 * s, -np.abs(d), d)
    d[~moving] = 0
    g = geom.copy()
    g[:, :3] += d
    return g


def cell_moves(geom, rng, exclude=()):
    """Spheres away from the hull moved by 0.7 of the spacing along one axis (most of a grid cell), the rest jittered by
    1 % of it inwards (inward_jitter)."""
    moving = ~np.isin(np.arange(len(geom)), list(exclude))
    s = spacing(geom[moving])
    g = inward_jitter(geom, rng, 0.01 * s, fixed=exclude)
    lo, hi = geom[moving, :3].min(0), geom[moving, :3].max(0)
    moved = []
    for i in range(len(g)):
        if i in exclude:
            continue
        axes = [k for k in range(3) if lo[k] + 1.01 * s <= geom[i, k] <= hi[k] - 1.01 * s]
        if axes and rng.random() < 0.3:
            k = axes[rng.integers(len(axes))]
            g[i, k] = geom[i, k] + F32(0.7 * s * (1 if rng.random() < 0.5 else -1))
            moved.append(i)
    return g, moved


def fresh(ctx, flat, cam):
    ctx.upload_flat(flat, cam)
    return ctx


def counters(st):
    return st.rays_primary, st.rays_shadow, st.rays_reflect


# ---- without a GPU ---------------------------------------------------------------------------------------------------------

def test_update_entry_points_are_exported():
    lib = _ffi.load()
    for name in ENTRY_POINTS:
        assert hasattr(lib, name), name


def test_update_entry_points_refuse_a_null_context():
    lib = _ffi.load()
    g = np.zeros((1, 4), F32)
    assert lib.tcrt_update_spheres(None, g.ctypes.data_as(C.c_void_p), None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_update_spheres_device(None, 0, g.ctypes.data_as(C.c_void_p), None) == _ffi.TCRT_ERR_INVALID


def test_sphere_geom_is_the_flattened_scene():
    rng = np.random.default_rng(3)
    centres = rng.uniform(-5, 5, (40, 3)).astype(F32)
    radii = rng.uniform(.01, 2.0, 40).astype(F32)
    radii[:3] = (F32(0.1), F32(1 / 3), F32(7.3))
    s = api.Scene()
    for c, r in zip(centres, radii):
        s.addSphere(tuple(float(v) for v in c), float(r))
    want = geom_of(s.flatten())
    got = api.sphere_geom(centres, radii)
    assert got.dtype == F32 and got.shape == (40, 4)
    assert (got.view(np.uint32) == want.view(np.uint32)).all()


def test_moved_flat_is_a_fresh_build():
    """moved_flat's edit of a flattened scene is what the host API builds from the moved spheres."""
    rng = np.random.default_rng(5)
    centres = rng.uniform(-3, 3, (30, 3)).astype(F32)
    radii = rng.uniform(.2, .5, 30).astype(F32)

    def scene(cs):
        s = api.Scene()
        s.addInfinitePlane((0, 0, -4), (0, 0, 1), (1, 0, 0))
        for k, (c, r) in enumerate(zip(cs, radii)):
            ref = s.addSphere(tuple(float(v) for v in c), float(r))
            if k % 10 == 0:
                ref.setAsLightSource(1.5)
        return s

    s0 = scene(centres)
    moved = centres + F32(0.25)
    s1 = scene(moved)
    f0, f1 = s0.flatten(), s1.flatten()
    m = moved_flat(f0, api.sphere_geom(moved, radii))
    n = f1.n_objects
    for name, width in (("sphere_geom", 4 * f1.n_spheres), ("obj_origin", 4 * n)):
        a = np.ctypeslib.as_array(getattr(m, name), (width,))
        b = np.ctypeslib.as_array(getattr(f1, name), (width,))
        assert (a.view(np.uint32) == b.view(np.uint32)).all(), name


# ---- on the GPU ------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def ref_ctx():
    """A second context for the fresh uploads the updated one is compared with."""
    ctx = api.Context([0])
    yield ctx
    ctx.close()


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


def _class(ctx):
    from test_kernel_variants import dispatch_class
    return dispatch_class(ctx.scene_structures())


def _variant_moves(name, flat, rng):
    """Jittered spheres and one light moved; in the room (fm1) one light outside the room, then back in."""
    g0 = geom_of(flat)
    lights = light_spheres(flat)
    g = inward_jitter(g0, rng, 0.02, fixed=lights)
    steps = []
    if VARIANTS[name][0] == "room":
        out = g.copy()
        out[lights[0], :3] = (ROOM_LO + ROOM_DIMS * np.array([.5, .5, 1.0]) + np.array([0, 0, 1.5])).astype(F32)
        steps.append(("light out of the room", out))
        back = g.copy()
        back[lights[0], :3] = g0[lights[0], :3] + F32(0.3)
        steps.append(("light back in", back))
    else:
        g[lights[0], :3] = g0[lights[0], :3] + np.array([.3, -.2, .1], F32)
        steps.append(("jitter and a light", g))
    return steps


@gpu
@pytest.mark.parametrize("depth", [0, 8, 64])
@pytest.mark.parametrize("name", NAMES)
def test_every_dispatch_class(gpu_ctx, ref_ctx, name, depth):
    s, cam = build(name)
    flat, c = s.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    cls = _class(gpu_ctx)
    rng = np.random.default_rng(depth + len(name))
    p = api.default_params(32, 24, depth)
    for what, g in _variant_moves(name, flat, rng):
        st = gpu_ctx.update_spheres(g)
        assert counters(st) == (0, 0, 0)
        assert _class(gpu_ctx) == cls, f"{name} {what}: the update changed the dispatch class"
        frame_pair(gpu_ctx, ref_ctx, moved_flat(flat, g), c, p, f"{name} {what} d{depth}", oracle=depth <= 8)


def _grid_scene(spec):
    if spec in VARIANTS:
        s, cam = build(spec)
    else:
        s, cam = make_scene(spec)
    return s, s.flatten(), cam.export()


def _aimed_rays(flat, geom, idx, eye):
    """From the eye: at each sphere's centre and just inside and outside its silhouette (1 -+ 1e-3 of the radius)."""
    dirs = []
    for i in idx:
        c, r = geom[i, :3].astype(np.float64), float(np.sqrt(max(float(geom[i, 3]), 0.0)))
        v = c - eye
        u = np.cross(v, [0.0, 0.0, 1.0])
        u = u / (np.linalg.norm(u) or 1.0)
        w = np.cross(v, u)
        w = w / (np.linalg.norm(w) or 1.0)
        dirs.append(v)
        for f in (1 - 1e-3, 1 + 1e-3):
            for a in (u, -u, w, -w):
                dirs.append(c + f * r * a - eye)
    return api.normalize_like_reference(np.asarray(dirs, F32))


@gpu
@pytest.mark.parametrize("spec", ["grid_fm0", "grid_fm3", "synth256", "lattice:3:8"])
def test_grid_kept_for_motion_inside_its_box(gpu_ctx, ref_ctx, rays_lib, spec):
    s, flat, c = _grid_scene(spec)
    gpu_ctx.upload_flat(flat, c)
    cells = gpu_ctx.scene_structures()["grid_cells"]
    assert cells > 0, spec
    rng = np.random.default_rng(11)
    g0 = geom_of(flat)
    gpu_ctx.update_spheres(g0)                 # the uploaded geometry itself: every registration as the builder made it
    assert gpu_ctx.scene_structures()["grid_cells"] == cells, spec
    g, moved = cell_moves(g0, rng, exclude=set(light_spheres(flat)))
    assert moved, spec
    gpu_ctx.update_spheres(g)
    assert gpu_ctx.scene_structures()["grid_cells"] == cells, spec
    m = moved_flat(flat, g)
    frame_pair(gpu_ctx, ref_ctx, m, c, api.default_params(64, 48, 6), spec, oracle=True)
    p = api.default_params(64, 48, 6)
    eye = np.array(c.eye[:], np.float64)
    dirs = _aimed_rays(m, g, moved, eye)
    o = np.array(c.eye[:], F32)
    got, bad, _ = gpu_ctx.intersect_rays(p, o, dirs)
    want, wbad = oracle_hits(rays_lib, m, p, o, dirs)
    assert bad == wbad == 0
    for k in HIT_NAMES:
        assert (np.asarray(got[k]).view(np.uint32) == np.asarray(want[k]).view(np.uint32)).all(), f"{spec} {k}"
    rgb, bad, _ = gpu_ctx.trace_rays(p, o, dirs)
    wrgb, _, _ = oracle_trace(rays_lib, m, p, o, dirs)
    assert (rgb.view(np.uint32) == wrgb.view(np.uint32)).all(), spec


@gpu
@pytest.mark.parametrize("spec", ["grid_fm0", "synth256"])
def test_grid_dropped_when_a_sphere_leaves_its_box(gpu_ctx, ref_ctx, spec):
    s, flat, c = _grid_scene(spec)
    gpu_ctx.upload_flat(flat, c)
    assert gpu_ctx.scene_structures()["grid_cells"] > 0
    cls = _class(gpu_ctx)
    g = geom_of(flat)
    i = next(k for k in range(len(g)) if k not in light_spheres(flat))
    g[i, 0] += F32(40.0)
    gpu_ctx.update_spheres(g)
    st = gpu_ctx.scene_structures()
    assert st["grid_cells"] == 0, spec
    assert _class(gpu_ctx) == ("render", 1, cls[2]), spec
    frame_pair(gpu_ctx, ref_ctx, moved_flat(flat, g), c, api.default_params(48, 32, 6), f"{spec} dropped")
    # it stays dropped through later updates, and a full upload brings it back
    gpu_ctx.update_spheres(geom_of(flat))
    assert gpu_ctx.scene_structures()["grid_cells"] == 0
    frame_pair(gpu_ctx, ref_ctx, flat, c, api.default_params(48, 32, 6), f"{spec} moved back")
    gpu_ctx.upload_flat(flat, c)
    assert gpu_ctx.scene_structures()["grid_cells"] > 0


@gpu
@pytest.mark.parametrize("spec", ["sb1_fm3", "grid_fm0", "synth256"])
def test_radii(gpu_ctx, ref_ctx, spec):
    s, flat, c = _grid_scene(spec)
    gpu_ctx.upload_flat(flat, c)
    g0 = geom_of(flat)
    lights = set(light_spheres(flat))
    plain = [i for i in range(len(g0)) if i not in lights]
    p = api.default_params(48, 32, 8)
    for what, i, r2 in (("3x radius", plain[len(plain) // 2], g0[plain[len(plain) // 2], 3] * F32(9)),
                        ("radius_squared 0", plain[1], F32(0)),
                        ("radius 1e-4", plain[2], F32(1e-8))):
        g = g0.copy()
        g[i, 3] = r2
        gpu_ctx.update_spheres(g)
        frame_pair(gpu_ctx, ref_ctx, moved_flat(flat, g), c, p, f"{spec} {what}", oracle=True)


@gpu
@pytest.mark.parametrize("name", ["sb1_fm1", "grid_fm0"])
def test_every_other_reader(gpu_ctx, ref_ctx, occ_lib, name):
    s, cam = build(name)
    flat, c = s.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    rng = np.random.default_rng(2)
    g = geom_of(flat)
    g[:, :3] += rng.normal(0, .03, (len(g), 3)).astype(F32)
    gpu_ctx.update_spheres(g)
    m = moved_flat(flat, g)
    fresh(ref_ctx, m, c)
    p = api.default_params(40, 32, 8)
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
    ha, _ = gpu_ctx.hit_buffers(p)
    hb, _ = ref_ctx.hit_buffers(p)
    for k in HIT_NAMES:
        assert (ha[k].view(np.uint32) == hb[k].view(np.uint32)).all(), k
    xs, zs = rng.integers(0, 40, 30), rng.integers(0, 32, 30)
    for x, y in zip(gpu_ctx.pick(p, xs, zs), ref_ctx.pick(p, xs, zs)):
        assert (x.view(np.uint32) == y.view(np.uint32)).all(), "pick"
    pts = np.concatenate([g[:, :3] + F32(.5), rng.uniform(-6, 6, (500, 3)).astype(F32)]).astype(F32)
    la, _, _ = gpu_ctx.occluded_lights(pts)
    lb, _, _ = ref_ctx.occluded_lights(pts)
    assert (la == lb).all(), "occluded_lights"
    want, _, _ = oracle_lights(occ_lib, m, pts)
    assert (la == want).all(), "occluded_lights vs oracle"
    o = np.array(c.eye[:], F32)
    d = api.normalize_like_reference(rng.normal(0, 1, (400, 3)).astype(F32))
    t = rng.uniform(.5, 20, 400).astype(F32)
    ra, _, _ = gpu_ctx.occluded_rays(o, d, t)
    rb, _, _ = ref_ctx.occluded_rays(o, d, t)
    assert (ra == rb).all(), "occluded_rays"
    from test_views import three_views
    va, sa = gpu_ctx.render_views(p, three_views(c))
    va = va.copy()
    vb, sb = ref_ctx.render_views(p, three_views(c))
    for v in range(3):
        assert_bit_identical(va[v], vb[v], f"view {v}")
    assert counters(sa) == counters(sb)
    assert gpu_ctx.balance_columns(p, 3) == ref_ctx.balance_columns(p, 3)


@gpu
def test_drift(gpu_ctx, ref_ctx):
    s, flat, c = _grid_scene("synth256")
    gpu_ctx.upload_flat(flat, c)
    rng = np.random.default_rng(30)
    g = geom_of(flat)
    lights = light_spheres(flat)
    step = 0.004 * spacing(np.delete(g, lights, 0))
    p = api.default_params(64, 48, 8)
    for k in range(1, 31):
        g = inward_jitter(g, rng, step, fixed=lights)
        gpu_ctx.update_spheres(g)
        assert gpu_ctx.scene_structures()["grid_cells"] > 0, k
        if k in (1, 10, 30):
            frame_pair(gpu_ctx, ref_ctx, moved_flat(flat, g), c, p, f"drift step {k}", oracle=k == 30)


@gpu
def test_ordering_and_the_upload_cache(gpu_ctx, ref_ctx):
    s, flat_a, c = _grid_scene("synth256")
    g_b = geom_of(flat_a)
    g_b[:, :3] += F32(0.05)
    flat_b = moved_flat(flat_a, g_b)
    p = api.default_params(64, 48, 6)
    want_a, _ = fresh(ref_ctx, flat_a, c).render(p)
    want_a = want_a.copy()
    want_b, _ = fresh(ref_ctx, flat_b, c).render(p)
    want_b = want_b.copy()
    bufs = [api.HostBuffer(64 * 48 * 12) for _ in range(3)]
    outs = [b.array(F32, (64, 48, 3)) for b in bufs]
    gpu_ctx.upload_flat(flat_a, c)
    t1 = gpu_ctx.render_async(p, out=outs[0])
    t2 = gpu_ctx.render_async(p, out=outs[1])
    gpu_ctx.update_spheres(g_b)
    gpu_ctx.wait(t1)
    t3 = gpu_ctx.render_async(p, out=outs[2])
    gpu_ctx.wait(t2)
    gpu_ctx.wait(t3)
    assert_bit_identical(outs[0], want_a, "frame 1")
    assert_bit_identical(outs[1], want_a, "frame 2")
    assert_bit_identical(outs[2], want_b, "frame 3")
    # an update makes the next upload rebuild: A again is A, B after updating to B is B
    gpu_ctx.upload_flat(flat_a, c)
    gpu_ctx.update_spheres(g_b)
    gpu_ctx.upload_flat(flat_a, c)
    assert_bit_identical(gpu_ctx.render(p)[0], want_a, "upload A after an update")
    gpu_ctx.update_spheres(g_b)
    gpu_ctx.upload_flat(flat_b, c)
    assert_bit_identical(gpu_ctx.render(p)[0], want_b, "upload B after updating to B")


@gpu
def test_errors(gpu_ctx):
    import torch

    s, flat, c = _grid_scene("sb1_fm0")
    gpu_ctx.upload_flat(flat, c)
    p = api.default_params(32, 24, 6)
    before, _ = gpu_ctx.render(p)
    before = before.copy()
    g0 = geom_of(flat)
    for k, v in ((0, np.nan), (1, np.inf), (2, -np.inf), (3, np.nan), (3, np.inf), (3, -1e-30)):
        g = g0 + F32(0.01)
        g[5, k] = F32(v)
        with pytest.raises(api.TcrtError) as e:
            gpu_ctx.update_spheres(g)
        assert e.value.code == _ffi.TCRT_ERR_INVALID
        t = torch.from_numpy(g).cuda()
        torch.cuda.synchronize()
        with pytest.raises(api.TcrtError) as e:
            gpu_ctx.update_spheres_device(t.data_ptr())
        assert e.value.code == _ffi.TCRT_ERR_INVALID
        assert_bit_identical(gpu_ctx.render(p)[0], before, f"after a refused update ({k}, {v})")
    with pytest.raises(api.TcrtError) as e:
        gpu_ctx.update_spheres_device(g0.ctypes.data)
    assert e.value.code == _ffi.TCRT_ERR_INVALID
    with pytest.raises(api.TcrtError) as e:
        gpu_ctx.update_spheres_device(0)
    assert e.value.code == _ffi.TCRT_ERR_INVALID
    new = api.Context([0])
    try:
        with pytest.raises(api.TcrtError) as e:
            new.update_spheres(g0)
        assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
        planes = api.Scene()
        planes.addInfinitePlane((0, 0, -1), (0, 0, 1), (1, 0, 0)).setCheckerBoard()
        planes.makeSceneBox((-3, -3, -2), (6, 6, 5))
        new.upload(planes, api.Camera())
        st = new.update_spheres(np.zeros((0, 4), F32))
        assert st.gpu_launches == 0
    finally:
        new.close()


@gpu
@pytest.mark.parametrize("spec", ["grid_fm0", "synth256"])
def test_a_refused_update_leaves_an_updated_grid_alone(gpu_ctx, ref_ctx, spec):
    """After a valid update the grid's item list lives in the update's own buffer; a refused update (host and device form)
    must not touch it, nor the cells, the spheres or the BVH.  The valid update moves spheres by most of a cell, so that
    cells list several spheres and a changed item list would show."""
    import torch

    s, flat, c = _grid_scene(spec)
    gpu_ctx.upload_flat(flat, c)
    cells = gpu_ctx.scene_structures()["grid_cells"]
    g, moved = cell_moves(geom_of(flat), np.random.default_rng(21), exclude=set(light_spheres(flat)))
    assert moved
    gpu_ctx.update_spheres(g)
    assert gpu_ctx.scene_structures()["grid_cells"] == cells, spec
    p = api.default_params(64, 48, 6)
    before = frame_pair(gpu_ctx, ref_ctx, moved_flat(flat, g), c, p, f"{spec} valid update")
    o = np.array(c.eye[:], F32)
    dirs = _aimed_rays(None, g, moved, o.astype(np.float64))
    hits_before, _, _ = gpu_ctx.intersect_rays(p, o, dirs)
    hits_before = {k: v.copy() for k, v in hits_before.items()}
    for k, v in ((0, np.nan), (3, -1.0), (2, np.inf)):
        bad = g + F32(0.02)
        bad[len(bad) // 2, k] = F32(v)
        with pytest.raises(api.TcrtError) as e:
            gpu_ctx.update_spheres(bad)
        assert e.value.code == _ffi.TCRT_ERR_INVALID
        t = torch.from_numpy(bad).cuda()
        torch.cuda.synchronize()
        with pytest.raises(api.TcrtError) as e:
            gpu_ctx.update_spheres_device(t.data_ptr())
        assert e.value.code == _ffi.TCRT_ERR_INVALID
        assert gpu_ctx.scene_structures()["grid_cells"] == cells, spec
        assert_bit_identical(gpu_ctx.render(p)[0], before, f"{spec} after a refused update ({k}, {v})")
        hits, _, _ = gpu_ctx.intersect_rays(p, o, dirs)
        for name in HIT_NAMES:
            assert (hits[name].view(np.uint32) == hits_before[name].view(np.uint32)).all(), f"{spec} {name}"


@gpu
def test_device_form_needs_16_byte_alignment(gpu_ctx):
    import torch

    s, flat, c = _grid_scene("synth256")
    gpu_ctx.upload_flat(flat, c)
    p = api.default_params(32, 24, 4)
    before = gpu_ctx.render(p)[0].copy()
    g = geom_of(flat)
    buf = torch.zeros(g.size + 4, dtype=torch.float32, device="cuda")
    buf[1:1 + g.size] = torch.from_numpy(g.ravel()).cuda()
    torch.cuda.synchronize()
    with pytest.raises(api.TcrtError) as e:
        gpu_ctx.update_spheres_device(buf.data_ptr() + 4)      # a float32 view one float into the buffer
    assert e.value.code == _ffi.TCRT_ERR_INVALID
    assert_bit_identical(gpu_ctx.render(p)[0], before, "after a misaligned pointer")
    buf[:g.size] = torch.from_numpy(g.ravel()).cuda()
    torch.cuda.synchronize()
    gpu_ctx.update_spheres_device(buf.data_ptr())
    assert_bit_identical(gpu_ctx.render(p)[0], before, "the uploaded geometry through the device form")


@gpu
def test_device_form_and_two_slots(gpu_ctx):
    import torch

    s, flat, c = _grid_scene("synth256")
    rng = np.random.default_rng(8)
    g, _ = cell_moves(geom_of(flat), rng, exclude=set(light_spheres(flat)))
    p = api.default_params(64, 48, 8)
    gpu_ctx.upload_flat(flat, c)
    gpu_ctx.update_spheres(g)
    want, st = gpu_ctx.render(p)
    want = want.copy()
    gpu_ctx.upload_flat(flat, c)
    t = torch.from_numpy(g).cuda()
    torch.cuda.synchronize()
    gpu_ctx.update_spheres_device(t.data_ptr())
    assert_bit_identical(gpu_ctx.render(p)[0], want, "device form")
    n_dev = api.device_count()
    pair = api.Context([0, 1 % n_dev])
    try:
        pair.upload_flat(flat, c)
        pair.update_spheres(g)
        img, st2 = pair.render(p)
        assert_bit_identical(img, want, "two slots, host form")
        assert counters(st2) == counters(st)
        for slot in (0, 1):
            pair.upload_flat(flat, c)
            with torch.cuda.device(pair.devices[slot]):
                ts = torch.from_numpy(g).cuda()
                torch.cuda.synchronize()
            pair.update_spheres_device(ts.data_ptr(), slot=slot)
            assert_bit_identical(pair.render(p)[0], want, f"two slots, device form from slot {slot}")
    finally:
        pair.close()
