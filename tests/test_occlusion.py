"""Occlusion queries (tcrt_occluded_rays, tcrt_occluded_lights and their device forms): the reference's shadow test
(inShadeCollisionDetection) for caller-supplied rays with their own limits, and its inShade for caller-supplied points
against every light.  Every answer is one the reference computes, so the calls are compared bit for bit, with their
counters, against the pinned oracle's own in_shade and shade_lights construction (tests/oracle_occlusion.c), and the
restatement itself is checked against the oracle's shadowed and unshadowed renders."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import make_scene
from test_kernel_variants import NAMES, VARIANTS, build as build_variant, dispatch_class
from test_ray_batches import GUARD, _upload_spec, crafted_rays, eye_rays, valid_rule

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
F32 = np.float32
INF = F32(np.inf)
FLT_MAX = np.finfo(F32).max
ENTRY_POINTS = ("tcrt_occluded_rays", "tcrt_occluded_lights", "tcrt_occluded_rays_device", "tcrt_occluded_lights_device")
PIECE = 1 << 22                 # rays or (point, light) pairs per piece (tcrt_api.cu kRayPiece)
# the named scenes and the dispatch class each must land in (the occlusion kernel serves every class; lattices walk
# their sphere BVH)
SCENES = {"default": ("render", 0, 1), "two_mirrors": ("render", 1, 3), "synth256": ("grid", 1, 0),
          "synth1024": ("grid", 1, 0), "boxes:3:14": ("render", 0, 2), "lattice:1:4": ("grid", 1, 0),
          "random:24:200": ("render", 1, 2)}


# ---- the oracle extension ---------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def occ_lib(tmp_path_factory):
    so = tmp_path_factory.mktemp("oracle_occlusion") / "liboracle_occlusion.so"
    subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared", "-ffp-contract=off",
                    os.path.join(ROOT, "tests", "oracle_occlusion.c"), "-o", str(so), "-lm"], check=True)
    lib = C.CDLL(str(so))
    ull = C.POINTER(C.c_ulonglong)
    lib.tcrt_oracle_occluded_rays.restype = C.c_int
    lib.tcrt_oracle_occluded_rays.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                              C.c_void_p, ull, ull]
    lib.tcrt_oracle_occluded_lights.restype = C.c_int
    lib.tcrt_oracle_occluded_lights.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, ull, ull]
    lib.tcrt_oracle_shadow_origins.restype = C.c_int
    lib.tcrt_oracle_shadow_origins.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    return lib


def _c(a):
    return np.ascontiguousarray(a, F32)


def oracle_rays(lib, flat, origins, dirs, tmax):
    """(occluded (n,) uint8, n_invalid, n_tests) of the oracle."""
    o, d, t = _c(origins), _c(dirs), _c(tmax)
    n = d.shape[0]
    out = np.empty(n, np.uint8)
    bad, tests = C.c_ulonglong(), C.c_ulonglong()
    assert lib.tcrt_oracle_occluded_rays(C.byref(flat), n, o.ctypes.data, int(o.shape == (3,)), d.ctypes.data, t.ctypes.data,
                                         out.ctypes.data, C.byref(bad), C.byref(tests)) == 0
    return out, int(bad.value), int(tests.value)


def oracle_lights(lib, flat, points):
    """(occluded (n, n_lights) uint8, n_invalid pairs, n_tests) of the oracle."""
    p = _c(points)
    n = p.shape[0]
    out = np.empty((n, flat.n_lights), np.uint8)
    bad, tests = C.c_ulonglong(), C.c_ulonglong()
    assert lib.tcrt_oracle_occluded_lights(C.byref(flat), n, p.ctypes.data, out.ctypes.data, C.byref(bad), C.byref(tests)) == 0
    return out, int(bad.value), int(tests.value)


def shadow_origins(lib, flat, cam, p):
    """(P (W*H, 3), kind (W*H,)) of the frame's eye rays: h.P of each primary hit; kind 1 non-light, 2 light, 0 miss."""
    n = p.width * p.height
    P = np.empty((n, 3), F32)
    kind = np.empty(n, np.uint8)
    assert lib.tcrt_oracle_shadow_origins(C.byref(flat), C.byref(cam), C.byref(p), 0, p.width, P.ctypes.data, kind.ctypes.data) == 0
    return P, kind


def light_positions(flat):
    org = np.ctypeslib.as_array(flat.obj_origin, (flat.n_objects * 4,)).reshape(-1, 4)[:, :3]
    return np.array([org[flat.light_obj[l]] for l in range(flat.n_lights)], F32).reshape(-1, 3)


def shadow_rays_like_reference(P, L):
    """The ray form of inShade(P, L) in numpy float32: lr = normalize_like_reference(L - P), dist = sqrt of the same
    unfused sum."""
    d = (L - P).astype(F32)
    with np.errstate(all="ignore"):
        dist = np.sqrt((d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2])
    return api.normalize_like_reference(d), dist.astype(F32)


def one_light(name):
    """(Scene, flat, camera) of `name` with only its first light left a light: the others stay as ordinary spheres."""
    s, cam = make_scene(name)
    flat = s.flatten()
    info = np.ctypeslib.as_array(flat.obj_info, (flat.n_objects * 4,)).reshape(-1, 4)
    for l in range(1, flat.n_lights):
        info[flat.light_obj[l], 2] = 0
    flat.n_lights = 1
    return s, flat, cam.export()


# ---- no device needed ------------------------------------------------------------------------------------------------

def test_occlusion_entry_points_are_exported():
    lib = _ffi.load()
    for name in ENTRY_POINTS:
        assert hasattr(lib, name), name


def test_occlusion_entry_points_refuse_a_null_context():
    lib = _ffi.load()
    o = np.zeros((4, 3), F32)
    d = np.tile(np.array([1, 0, 0], F32), (4, 1))
    t = np.ones(4, F32)
    out = np.full(4, 7, np.uint8)
    bad = C.c_ulonglong(99)
    st = _ffi.TcrtStats()
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    assert lib.tcrt_occluded_rays(None, 4, ptr(o), 0, ptr(d), ptr(t), ptr(out), C.byref(bad), C.byref(st)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_rays(None, 0, None, 0, None, None, None, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_lights(None, 4, ptr(o), ptr(out), C.byref(bad), C.byref(st)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_lights(None, 1 << 62, ptr(o), ptr(out), None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_rays_device(None, 0, 4, ptr(o), 0, ptr(d), ptr(t), ptr(out), None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_lights_device(None, -1, 4, ptr(o), ptr(out), None, None) == _ffi.TCRT_ERR_INVALID
    assert bad.value == 99 and (out == 7).all()


@pytest.mark.parametrize("name", ["default", "boxes:3:14", "lattice:1:4", "random:24:200"])
def test_restatement_agrees_with_the_reference_renders(occ_lib, name):
    """One-light scenes, reflections off: at every non-light primary hit the restated inShade decides the pixel.  Where it
    says occluded the shadowed pixel is exactly (+0, +0, +0); where not, it equals the unshadowed pixel bit for bit."""
    s, flat, c = one_light(name)
    w, h = 96, 72
    on = api.default_params(w, h, 0, shadows=True, reflections=False)
    off = api.default_params(w, h, 0, shadows=False, reflections=False)
    img_on, _ = O.render(flat, c, on)
    img_off, _ = O.render(flat, c, off)
    img_on, img_off = img_on.reshape(-1, 3), img_off.reshape(-1, 3)
    P, kind = shadow_origins(occ_lib, flat, c, on)
    hit = kind == 1
    occl, n_bad, n_tests = oracle_lights(occ_lib, flat, P[hit])
    assert n_bad == 0 and n_tests == int(hit.sum())
    occl = occl[:, 0]
    shadowed = img_on[hit][occl == 1].view(np.uint32)
    lit_on, lit_off = img_on[hit][occl == 0].view(np.uint32), img_off[hit][occl == 0].view(np.uint32)
    assert len(shadowed) > 0 and len(lit_on) > 0, (len(shadowed), len(lit_on))
    assert (shadowed == 0).all(), "an occluded pixel is not (+0, +0, +0)"
    assert np.array_equal(lit_on, lit_off), "an unoccluded pixel differs from the unshadowed frame"
    assert (lit_on != 0).any(), "no lit pixel is non-zero"


def test_tmax_rule_at_its_boundaries(occ_lib):
    """tmax -0, +0 and NaN are refused; the smallest denormal, FLT_MAX and +inf are traced."""
    s, cam = make_scene("default")
    flat = s.flatten()
    eye = np.array(cam.export().eye[:], F32)
    d = np.tile(api.normalize_like_reference(np.array([[0.2, 1.0, -0.1]], F32)), (6, 1))
    t = np.array([-0.0, 0.0, np.nan, np.nextafter(F32(0), F32(1)), FLT_MAX, np.inf], F32)
    out, n_bad, n_tests = oracle_rays(occ_lib, flat, eye, d, t)
    assert list(out[:3]) == [0xFF] * 3 and n_bad == 3 and n_tests == 3
    assert out[3] == 0 and out[4] == out[5] and out[4] in (0, 1)
    # the batch rule still applies: the crafted rays with tmax = inf
    o, dd, valid = crafted_rays()
    out, n_bad, _ = oracle_rays(occ_lib, flat, o, dd, np.full(len(o), INF))
    assert ((out == 0xFF) == ~valid).all() and n_bad == int((~valid).sum())


def test_points_at_and_near_a_light(occ_lib):
    """A point exactly at a light is an invalid pair (the reference's 0/0 would say "not in shade"); one a few ulps away
    is a valid pair.  The 2^40 origin boundary holds for points, and refuses the whole row."""
    s, cam = make_scene("default")
    flat = s.flatten()
    L = light_positions(flat)
    near = np.array([np.nextafter(L[0], F32(np.inf)), L[0] + np.spacing(L[0]) * 4, L[0] - np.spacing(L[0]) * 3], F32)
    big = F32(2.0 ** 40)
    pts = np.concatenate([L[:1], near, [[big, -big, big], [np.nextafter(big, INF), 0, 0], [np.nan, 0, 0]]]).astype(F32)
    out, n_bad, n_tests = oracle_lights(occ_lib, flat, pts)
    nl = flat.n_lights
    assert out[0, 0] == 0xFF and (out[0, 1:] != 0xFF).all()
    assert (out[1:4] != 0xFF).all()
    assert (out[4] != 0xFF).all() and (out[5:] == 0xFF).all()
    assert n_bad == 1 + 2 * nl and n_tests == len(pts) * nl - n_bad


@pytest.mark.parametrize("name", ["default", "boxes:3:14", "lattice:1:4"])
def test_ray_form_of_the_numpy_recipe_is_the_points_form(occ_lib, name):
    s, cam = make_scene(name)
    flat = s.flatten()
    rng = np.random.default_rng(3)
    L = light_positions(flat)
    pts = rng.uniform(-6, 6, (2000, 3)).astype(F32)
    want, _, _ = oracle_lights(occ_lib, flat, pts)
    for l in range(flat.n_lights):
        lr, dist = shadow_rays_like_reference(pts, np.broadcast_to(L[l], pts.shape))
        got, n_bad, _ = oracle_rays(occ_lib, flat, pts, lr, dist)
        assert n_bad == 0 and np.array_equal(got, want[:, l]), f"light {l}"
    assert (want == 1).any() and (want == 0).any()


# ---- on the GPU ------------------------------------------------------------------------------------------------------

def _stats_ok(st, n_tests, launches=None):
    assert st.rays_shadow == n_tests and st.rays_primary == 0 and st.rays_reflect == 0, (st.rays_shadow, n_tests)
    if launches is not None:
        assert st.gpu_launches == launches


def check_lights(ctx, lib, flat, pts, what):
    want, w_bad, w_tests = oracle_lights(lib, flat, pts)
    got, g_bad, st = ctx.occluded_lights(_c(pts))
    assert got.shape == want.shape, what
    bad = int((got != want).any(-1).sum())
    assert bad == 0, f"{what}: {bad} of {len(pts)} points differ"
    assert g_bad == w_bad, what
    _stats_ok(st, w_tests)
    return got


def check_rays(ctx, lib, flat, o, d, t, what):
    want, w_bad, w_tests = oracle_rays(lib, flat, o, d, t)
    got, g_bad, st = ctx.occluded_rays(_c(o), _c(d), _c(t))
    bad = int((got != want).sum())
    assert bad == 0, f"{what}: {bad} of {len(d)} rays differ"
    assert g_bad == w_bad, what
    _stats_ok(st, w_tests)
    return got


def scene_points(ctx, lib, flat, c, rng):
    """Points in and around the scene: the eye rays' shadow-ray origins, random points in its box, inside spheres, within
    a few cluster margins of every box-cluster wall on both sides (with the grazing light's wall), and 600, 1e6 and 2^40
    away."""
    P, kind = shadow_origins(lib, flat, c, api.default_params(64, 48, 0))
    parts = [P[kind == 1]]
    n_s = flat.n_spheres
    sph = np.ctypeslib.as_array(flat.sphere_geom, (n_s * 4,)).reshape(n_s, 4) if n_s else np.zeros((0, 4), F32)
    eye = np.array(c.eye[:], F32)
    lo = np.minimum(sph[:, :3].min(0) if n_s else eye, eye) - 2
    hi = np.maximum(sph[:, :3].max(0) if n_s else eye, eye) + 2
    parts.append(rng.uniform(lo, hi, (2048, 3)).astype(F32))
    if n_s:
        k = rng.integers(0, n_s, 512)
        parts.append(sph[k, :3] + rng.uniform(-.5, .5, (512, 3)).astype(F32) * np.sqrt(sph[k, 3:4]))
    # walls: every finite and infinite plane, points at +-{0.5, 1, 2, 4} x 1e-5 x |coordinate| and at +-1e-3 along its normal
    for geom, count in ((flat.fin_geom, flat.n_fin_planes), (flat.inf_geom, flat.n_inf_planes)):
        if not count:
            continue
        g = np.ctypeslib.as_array(geom, (count * 16,)).reshape(count, 16)
        org, nrm = g[:, 12:15], g[:, 0:3]
        if geom is flat.fin_geom:      # a point of the rectangle
            u, v = (rng.uniform(0, 1, (count, 1)) * g[:, k:k + 1] for k in (7, 11))
        else:                          # a point of the plane near its origin
            u, v = rng.uniform(-3, 3, (2, count, 1))
        base = (org + g[:, 4:7] * u.astype(F32) + g[:, 8:11] * v.astype(F32)).astype(F32)
        for off in (0.5e-5, 1e-5, 2e-5, 4e-5, 1e-3, 0.5e-3):
            for sgn in (1, -1):
                parts.append((base + nrm * F32(sgn * off * max(1.0, float(np.abs(base).max())))).astype(F32))
    for r in (600.0, 1e6, 2.0 ** 40):
        far = api.normalize_like_reference(rng.standard_normal((256, 3)).astype(F32)) * F32(r)
        parts.append(np.clip(far, -F32(2.0 ** 40), F32(2.0 ** 40)))
    L = light_positions(flat)
    parts.append(L)                                   # points at the lights: invalid pairs
    parts.append(L + np.spacing(L) * 2)
    return np.ascontiguousarray(np.concatenate(parts), F32)


def scene_rays(ctx, lib, flat, c, rng):
    """(origins, directions, tmax) of the ray form: random rays with +inf and FLT_MAX, the tie boundary of every ray whose
    nearest hit is a non-light at d > 0 (tmax = d: 0, next float: 1), and rays aimed through a light at a light behind
    it."""
    n_s = flat.n_spheres
    sph = np.ctypeslib.as_array(flat.sphere_geom, (n_s * 4,)).reshape(n_s, 4) if n_s else np.zeros((0, 4), F32)
    eye = np.array(c.eye[:], F32)
    lo = np.minimum(sph[:, :3].min(0) if n_s else eye, eye) - 2
    hi = np.maximum(sph[:, :3].max(0) if n_s else eye, eye) + 2
    o = rng.uniform(lo, hi, (4096, 3)).astype(F32)
    d = api.normalize_like_reference(rng.standard_normal((4096, 3)).astype(F32))
    o_e, d_e, _ = eye_rays(c, 64, 48)
    o = np.concatenate([o, o_e])
    d = np.concatenate([d, d_e])
    hits, _, _ = ctx.intersect_rays(api.default_params(1, 1, 0), o, d)
    info = np.ctypeslib.as_array(flat.obj_info, (flat.n_objects * 4,)).reshape(-1, 4)
    obj, dist = hits["object"], hits["distance"]
    tie = (obj >= 0) & (dist > 0)
    tie[tie] &= info[obj[tie], 2] == 0
    ot, dt, t = [o, o], [d, d], [np.full(len(d), INF), np.full(len(d), FLT_MAX)]
    ot += [o[tie], o[tie]]
    dt += [d[tie], d[tie]]
    t += [dist[tie], np.nextafter(dist[tie], INF)]
    L = light_positions(flat)
    through = []
    for a in range(len(L)):
        for b in range(len(L)):
            if a != b:
                u = api.normalize_like_reference((L[a] - L[b])[None])[0]
                src = L[a] + u * F32(1.0) + rng.uniform(-.05, .05, (64, 3)).astype(F32)
                lr, dd = shadow_rays_like_reference(src, np.broadcast_to(L[b], src.shape))
                through.append((src, lr, dd))
    for src, lr, dd in through:
        ot.append(src)
        dt.append(lr)
        t.append(dd)
    return (np.ascontiguousarray(np.concatenate(ot), F32), np.ascontiguousarray(np.concatenate(dt), F32),
            np.ascontiguousarray(np.concatenate(t), F32), int(tie.sum()), len(through) * 64)


def check_scene(ctx, lib, flat, c, seed, what):
    rng = np.random.default_rng(seed)
    pts = scene_points(ctx, lib, flat, c, rng)
    got = check_lights(ctx, lib, flat, pts, f"{what} points")
    assert (got == 1).any() and (got == 0).any() and (got == 0xFF).any(), what
    o, d, t, n_tie, n_through = scene_rays(ctx, lib, flat, c, rng)
    got = check_rays(ctx, lib, flat, o, d, t, f"{what} rays")
    n = (len(o) - 2 * n_tie - n_through) // 2
    tie = got[2 * n:2 * n + 2 * n_tie]
    assert (tie[:n_tie] == 0).all() and (tie[n_tie:] == 1).all(), f"{what}: tie boundary"
    assert n_tie > 100, (what, n_tie)
    return got, o, d, n_through


@gpu
@pytest.mark.parametrize("name", NAMES)
def test_every_dispatch_class_matches_the_oracle(gpu_ctx, occ_lib, name):
    s, cam = build_variant(name)
    flat, c = s.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    assert dispatch_class(gpu_ctx.scene_structures()) == VARIANTS[name][3]
    got, o, d, n_through = check_scene(gpu_ctx, occ_lib, flat, c, NAMES.index(name), name)
    # the rays aimed through a light at the light behind it: lights never block
    through = slice(len(o) - n_through, len(o))
    h, _, _ = gpu_ctx.intersect_rays(api.default_params(1, 1, 0), o[through], d[through])
    info = np.ctypeslib.as_array(flat.obj_info, (flat.n_objects * 4,)).reshape(-1, 4)
    first_is_light = (h["object"] >= 0) & (info[np.maximum(h["object"], 0), 2] != 0)
    assert (first_is_light & (got[through] == 0)).any(), "no ray passed a light unblocked"


@gpu
@pytest.mark.parametrize("spec", list(SCENES))
def test_named_scenes_match_the_oracle(gpu_ctx, occ_lib, spec):
    s, flat, c = _upload_spec(gpu_ctx, spec)
    assert dispatch_class(gpu_ctx.scene_structures()) == SCENES[spec]
    check_scene(gpu_ctx, occ_lib, flat, c, hash(spec) % 1000, spec)


@gpu
def test_mixed_invalid_inputs(gpu_ctx, occ_lib):
    for spec in ("synth256", "default"):
        s, flat, c = _upload_spec(gpu_ctx, spec)
        rng = np.random.default_rng(11)
        o_v, d_v, _ = eye_rays(c, 32, 24, "shuffle")
        o_x, d_x, valid_x = crafted_rays()
        o = np.concatenate([o_v, o_x, o_v[:5]])
        d = np.concatenate([d_v, d_x, d_v[:5]])
        t = np.full(len(o), INF)
        t[rng.choice(len(o), 40, replace=False)] = F32(np.nan)
        t[rng.choice(len(o), 40, replace=False)] = F32(-0.0)
        t[rng.choice(len(o), 40, replace=False)] = F32(0.0)
        t[rng.choice(len(o), 40, replace=False)] = np.nextafter(F32(0), F32(1))
        got = check_rays(gpu_ctx, occ_lib, flat, o, d, t, f"{spec} mixed rays")
        assert ((got == 0xFF) == ~(valid_rule(o, d) & (t > 0))).all()
        pts = np.concatenate([o_v[:1] + d_v * F32(2), [[np.nan, 0, 0], [0, np.inf, 0], [F32(2.0 ** 41), 0, 0]],
                              light_positions(flat)]).astype(F32)
        check_lights(gpu_ctx, occ_lib, flat, pts, f"{spec} mixed points")
        # all invalid
        got, n_bad, st = gpu_ctx.occluded_rays(o_x[~valid_x], d_x[~valid_x], np.ones(int((~valid_x).sum()), F32))
        assert (got == 0xFF).all() and n_bad == len(got) and st.rays_shadow == 0


@gpu
@pytest.mark.parametrize("n", [0, 1, 31, 33])
def test_small_batches(gpu_ctx, occ_lib, n):
    s, flat, c = _upload_spec(gpu_ctx, "two_mirrors")
    o, d, _ = eye_rays(c, 16, 8, "shuffle")
    o, d = o[:n], d[:n]
    t = np.full(n, F32(5.0))
    got, _, st = gpu_ctx.occluded_rays(o, d, t)
    want, _, tests = oracle_rays(occ_lib, flat, o, d, t)
    assert np.array_equal(got, want)
    _stats_ok(st, tests, 1 if n else 0)
    pts = o + d * F32(3)
    got, _, st = gpu_ctx.occluded_lights(_c(pts))
    want, _, tests = oracle_lights(occ_lib, flat, pts)
    assert np.array_equal(got, want)
    _stats_ok(st, tests, 1 if n else 0)


@gpu
def test_a_scene_without_lights(gpu_ctx, occ_lib):
    s = api.Scene()
    s.addSphere((0, 5, 0), 1.0)
    cam = api.Camera()
    gpu_ctx.upload(s, cam)
    flat = s.flatten()
    got, n_bad, st = gpu_ctx.occluded_lights(np.zeros((10, 3), F32))
    assert got.shape == (10, 0) and n_bad == 0 and st.gpu_launches == 0
    d = np.tile(np.array([[0, 1, 0]], F32), (3, 1))
    got = check_rays(gpu_ctx, occ_lib, flat, np.zeros((3, 3), F32), d, np.array([3.0, 4.0, 4.5], F32), "no lights")
    assert list(got) == [0, 0, 1]


@gpu
def test_batches_of_several_pieces(gpu_ctx, occ_lib):
    """Rays: the 4K eye rays (8.3 M, two pieces) and 1.5x that (three pieces on three render streams) with tmax = +inf.
    Points: 4.5 M points x 2 lights (3 pieces of 2 Mi points).  Each against the same items in single-piece calls, and
    against the oracle around every piece boundary."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    flat, c = scene.flatten(), cam.export()
    o, d, _ = eye_rays(c, 3840, 2160)
    m = len(o)
    o2, d2 = np.concatenate([o, o[:m // 2]]), np.concatenate([d, d[:m // 2]])
    t = np.full(len(o2), INF)
    got, n_bad, st = gpu_ctx.occluded_rays(o2, d2, t)
    got = got.copy()
    assert n_bad == 0 and st.gpu_launches == 3
    step = PIECE // 2
    ref = np.concatenate([gpu_ctx.occluded_rays(o2[a:a + step], d2[a:a + step], t[a:a + step])[0].copy()
                          for a in range(0, len(o2), step)])
    assert np.array_equal(got, ref)
    for b in range(PIECE, len(o2), PIECE):
        want, _, _ = oracle_rays(occ_lib, flat, o2[b - 64:b + 64], d2[b - 64:b + 64], t[b - 64:b + 64])
        assert np.array_equal(got[b - 64:b + 64], want), f"piece boundary {b}"
    per = PIECE // flat.n_lights
    pts = _c(o2[:int(2.2 * per)] + d2[:int(2.2 * per)] * F32(4))
    got, n_bad, st = gpu_ctx.occluded_lights(pts)
    got = got.copy()
    assert st.gpu_launches == 3 and st.rays_shadow == len(pts) * flat.n_lights - n_bad
    ref = np.concatenate([gpu_ctx.occluded_lights(pts[a:a + per // 2])[0].copy() for a in range(0, len(pts), per // 2)])
    assert np.array_equal(got, ref)
    for b in range(per, len(pts), per):
        want, _, _ = oracle_lights(occ_lib, flat, pts[b - 64:b + 64])
        assert np.array_equal(got[b - 64:b + 64], want), f"points piece boundary {b}"


@gpu
def test_destinations(gpu_ctx):
    """Pinned and pageable inputs and outputs (with guard words), and the device forms with torch tensors: identical."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    o, d, _ = eye_rays(c, 1024, 768, "tile")          # 786 K rays: the staged copy-out of pageable outputs
    n = len(o)
    t = np.full(n, F32(7.5))
    pts = _c(o + d * F32(3))
    ref, _, st_ref = gpu_ctx.occluded_rays(o, d, t)
    ref = ref.copy()
    ref_l, _, st_l = gpu_ctx.occluded_lights(pts)
    ref_l = ref_l.copy()
    nl = ref_l.shape[1]
    bufs = []

    def pinned(nbytes):
        hb = api.HostBuffer(nbytes + 2 * GUARD * 4)
        bufs.append(hb)
        a = hb.array(np.uint8, (hb.nbytes,))
        a[:] = 0xAB
        return a[4 * GUARD:4 * GUARD + nbytes], a

    def pageable(nbytes):
        a = np.full(nbytes + 8 * GUARD, 0xAB, np.uint8)
        return a[4 * GUARD:len(a) - 4 * GUARD], a

    for in_kind in (pinned, pageable):
        oi = in_kind(o.nbytes)[0].view(F32).reshape(n, 3)
        di = in_kind(d.nbytes)[0].view(F32).reshape(n, 3)
        ti = in_kind(t.nbytes)[0].view(F32)
        pi = in_kind(pts.nbytes)[0].view(F32).reshape(n, 3)
        oi[:], di[:], ti[:], pi[:] = o, d, t, pts
        for out_kind in (pinned, pageable):
            out, whole = out_kind(n)
            got, _, st = gpu_ctx.occluded_rays(oi, di, ti, out=out)
            assert np.array_equal(got, ref), f"{in_kind.__name__} -> {out_kind.__name__}"
            assert (whole[:4 * GUARD] == 0xAB).all() and (whole[-4 * GUARD:] == 0xAB).all()
            assert st.rays_shadow == st_ref.rays_shadow
            out, whole = out_kind(n * nl)
            got, _, st = gpu_ctx.occluded_lights(pi, out=out.reshape(n, nl))
            assert np.array_equal(got, ref_l), f"points {in_kind.__name__} -> {out_kind.__name__}"
            assert (whole[:4 * GUARD] == 0xAB).all() and (whole[-4 * GUARD:] == 0xAB).all()
            assert st.rays_shadow == st_l.rays_shadow
    import torch
    dev = torch.device("cuda:0")
    to, td, tt, tp = (torch.from_numpy(a).to(dev) for a in (o, d, t, pts))
    tout = torch.full((n + 64,), 0xAB, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    n_bad, st = gpu_ctx.occluded_rays_device(n, to.data_ptr(), td.data_ptr(), tt.data_ptr(), tout.data_ptr())
    res = tout.cpu().numpy()
    assert n_bad == 0 and st.rays_shadow == st_ref.rays_shadow
    assert np.array_equal(res[:n], ref) and (res[n:] == 0xAB).all()
    tshared = torch.from_numpy(o[0].copy()).to(dev)
    torch.cuda.synchronize()
    gpu_ctx.occluded_rays_device(n, tshared.data_ptr(), td.data_ptr(), tt.data_ptr(), tout.data_ptr(), shared_origin=True)
    assert np.array_equal(tout.cpu().numpy()[:n], ref), "device form, shared origin"
    tl = torch.full((n * nl + 64,), 0xAB, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    n_bad, st = gpu_ctx.occluded_lights_device(n, tp.data_ptr(), tl.data_ptr())
    res = tl.cpu().numpy()
    assert np.array_equal(res[:n * nl].reshape(n, nl), ref_l) and (res[n * nl:] == 0xAB).all()
    assert st.rays_shadow == st_l.rays_shadow
    with pytest.raises(api.TcrtError) as e:
        gpu_ctx.occluded_rays_device(n, to.data_ptr(), td.data_ptr(), tt.data_ptr(), tout.data_ptr(), slot=1)
    assert e.value.code == _ffi.TCRT_ERR_INVALID
    with pytest.raises(api.TcrtError) as e:
        gpu_ctx.occluded_rays_device(n, to.data_ptr(), td.data_ptr(), t.ctypes.data, tout.data_ptr())
    assert e.value.code == _ffi.TCRT_ERR_INVALID
    with pytest.raises(api.TcrtError) as e:
        gpu_ctx.occluded_lights_device(n, pts.ctypes.data, tl.data_ptr())
    assert e.value.code == _ffi.TCRT_ERR_INVALID


@gpu
def test_error_codes(gpu_ctx):
    lib = _ffi.load()
    o = np.zeros((4, 3), F32)
    d = np.tile(np.array([1, 0, 0], F32), (4, 1))
    t = np.ones(4, F32)
    out = np.empty(16, np.uint8)
    fresh = api.Context([0])
    with pytest.raises(api.TcrtError) as e:
        fresh.occluded_rays(o, d, t)
    assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    assert lib.tcrt_occluded_lights(fresh._h, 4, ptr(o), ptr(out), None, None) == _ffi.TCRT_ERR_NO_SCENE
    fresh.close()
    _upload_spec(gpu_ctx, "default")
    h = gpu_ctx._h
    assert lib.tcrt_occluded_rays(h, 4, ptr(o), 0, ptr(d), ptr(t), None, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_rays(h, 4, None, 0, ptr(d), ptr(t), ptr(out), None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_rays(h, 4, ptr(o), 0, None, ptr(t), ptr(out), None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_rays(h, 4, ptr(o), 0, ptr(d), None, ptr(out), None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_rays(h, 1 << 62, ptr(o), 0, ptr(d), ptr(t), ptr(out), None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_lights(h, 4, None, ptr(out), None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_lights(h, 4, ptr(o), None, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_lights(h, 1 << 62, ptr(o), ptr(out), None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_occluded_rays(h, 0, None, 0, None, None, ptr(out), None, None) == _ffi.TCRT_OK
    assert lib.tcrt_occluded_lights(h, 0, None, ptr(out), None, None) == _ffi.TCRT_OK


@gpu
def test_queries_leave_the_last_render_and_the_camera_alone(gpu_ctx, occ_lib, tmp_path):
    scene, cam = make_scene("two_mirrors")
    gpu_ctx.upload(scene, cam)
    flat, c = scene.flatten(), cam.export()
    p = api.default_params(64, 48, 20)
    frame, _ = gpu_ctx.render(p)
    frame = frame.copy()
    gpu_ctx.write_ppm(p, str(tmp_path / "a.ppm"))
    o, d, _ = eye_rays(c, 64, 48)
    t = np.full(len(o), INF)
    P, kind = shadow_origins(occ_lib, flat, c, api.default_params(64, 48, 0))
    pts = _c(P[kind == 1])
    ref, _, _ = gpu_ctx.occluded_rays(o, d, t)
    ref = ref.copy()
    ref_l, _, _ = gpu_ctx.occluded_lights(pts)
    ref_l = ref_l.copy()
    buf = [api.HostBuffer(64 * 48 * 12) for _ in range(2)]
    outs = [b.array(F32, (64, 48, 3)) for b in buf]
    tk = [gpu_ctx.render_async(p, 0, 64, outs[k]) for k in range(2)]
    got, _, _ = gpu_ctx.occluded_rays(o, d, t)
    assert np.array_equal(got, ref), "with two frames in flight"
    got, _, _ = gpu_ctx.occluded_lights(pts)
    assert np.array_equal(got, ref_l), "points with two frames in flight"
    for k in range(2):
        gpu_ctx.wait(tk[k])
        assert np.array_equal(outs[k].view(np.uint32), frame.view(np.uint32)), "frame in flight"
    assert np.array_equal(gpu_ctx.download(np.empty_like(frame)).view(np.uint32), frame.view(np.uint32)), "last render"
    gpu_ctx.write_ppm(p, str(tmp_path / "b.ppm"))
    assert (tmp_path / "a.ppm").read_bytes() == (tmp_path / "b.ppm").read_bytes()
    c2 = cam.export()
    for k in range(3):
        c2.eye[k] += 0.5
        c2.screen_origin[k] += 0.5
    gpu_ctx.set_camera(c2)
    got, _, _ = gpu_ctx.occluded_rays(o, d, t)
    assert np.array_equal(got, ref), "after tcrt_set_camera"
    got, _, _ = gpu_ctx.occluded_lights(pts)
    assert np.array_equal(got, ref_l), "points after tcrt_set_camera"


@gpu
@pytest.mark.parametrize("n_bands", [2, 3])
def test_multi_device_queries(gpu_ctx, n_bands):
    n_dev = api.device_count()
    scene, cam = make_scene("synth256")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    o, d, _ = eye_rays(c, 320, 240, "tile")
    t = np.full(len(o), F32(30.0))
    pts = _c(o + d * F32(5))
    ref, _, st1 = gpu_ctx.occluded_rays(o, d, t)
    ref = ref.copy()
    ref_l, _, st1l = gpu_ctx.occluded_lights(pts)
    ref_l = ref_l.copy()
    multi = api.Context([i % n_dev for i in range(n_bands)])
    multi.upload(scene, cam)
    n = len(o)
    got, _, st = multi.occluded_rays(o, d, t)
    assert np.array_equal(got, ref)
    assert st.bands == [(n * i // n_bands, n * (i + 1) // n_bands) for i in range(n_bands)]
    assert st.rays_shadow == st1.rays_shadow
    got, _, st = multi.occluded_lights(pts)
    assert np.array_equal(got, ref_l)
    assert st.bands == [(n * i // n_bands, n * (i + 1) // n_bands) for i in range(n_bands)]
    assert st.rays_shadow == st1l.rays_shadow
    multi.close()


CPP_PROGRAM = r"""
#include <math.h>
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
    const int W = 48, H = 36;
    std::vector<Ray> rays;
    std::vector<float> tmax;
    std::vector<vector3d> points;
    for (int x = 0; x < W; x++)
        for (int z = 0; z < H; z++) {
            Ray* r = camera.createEyeRay(((float)x) / W, ((float)z) / H);
            rays.push_back(*r);
            tmax.push_back(INFINITY);
            vector3d o = r->getOrigin(), d = r->getDirection();
            points.push_back(vector3d(o.x + d.x * 3.0f, o.y + d.y * 3.0f, o.z + d.z * 3.0f));
            delete r;
        }
    GpuRayTracer rt;
    std::vector<unsigned char> occ(rays.size()), occ_l(points.size() * 8);
    unsigned long long bad = 99, bad_l = 99;
    if (!rt.ok() || rt.setScene(scene, camera) || rt.occludedRays(rays, tmax, occ.data(), &bad) ||
        rt.occludedLights(points, occ_l.data(), &bad_l)) {
        fprintf(stderr, "%s\n", rt.lastError());
        return 1;
    }
    if (rt.occludedRays(rays, std::vector<float>(3, 1.0f), occ.data()) != TCRT_ERR_INVALID) return 1;
    printf("%llu %llu\n", bad, bad_l);
    FILE* f = fopen("occ.bin", "wb");
    if (!f) return 1;
    fwrite(occ.data(), 1, occ.size(), f);
    fwrite(occ_l.data(), 1, occ_l.size(), f);
    return fclose(f) ? 1 : 0;
}
"""


@gpu
def test_cpp_occlusion(gpu_ctx, tmp_path):
    src = tmp_path / "occ.cpp"
    src.write_text(CPP_PROGRAM)
    libdir = os.path.join(ROOT, "tilecoderaytracer_b200")
    exe = tmp_path / "occ"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), str(src),
                    "-L", libdir, "-ltcrt", f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.split() == ["0", "0"]
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    o, d, _ = eye_rays(cam.export(), 48, 36)
    n = len(o)
    raw = np.fromfile(tmp_path / "occ.bin", dtype=np.uint8)
    want, _, _ = gpu_ctx.occluded_rays(o, d, np.full(n, INF))
    assert np.array_equal(raw[:n], want)
    pts = _c(o + d * F32(3))
    want_l, _, _ = gpu_ctx.occluded_lights(pts)
    assert np.array_equal(raw[n:n + want_l.size], want_l.ravel())
