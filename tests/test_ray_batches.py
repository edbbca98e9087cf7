"""Ray batches (tcrt_trace_rays, tcrt_intersect_rays and their device forms): the colour and the nearest hit of
caller-supplied rays, computed by the render and hit kernels' ray mode.  Every value is one the reference computes for a
Ray holding exactly the given origin and direction, so batches are compared bit for bit with the pinned oracle's own
trace_pixel and nearest_hit (tests/oracle_rays.c), and a frame's eye rays must reproduce the frame."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import assert_bit_identical, bits, make_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
HIT_NAMES = ("object", "distance", "normal")
ENTRY_POINTS = ("tcrt_trace_rays", "tcrt_intersect_rays", "tcrt_trace_rays_device", "tcrt_intersect_rays_device")
PIECE = 1 << 22                 # rays per piece (tcrt_api.cu kRayPiece)
F32 = np.float32


# ---- the oracle extension and the numpy restatements -------------------------------------------------------------------

@pytest.fixture(scope="module")
def rays_lib(tmp_path_factory):
    so = tmp_path_factory.mktemp("oracle_rays") / "liboracle_rays.so"
    subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", os.path.join(ROOT, "tests", "oracle_rays.c"),
                    "-o", str(so), "-lm"], check=True)
    lib = C.CDLL(str(so))
    lib.tcrt_oracle_ray_valid.restype = C.c_int
    lib.tcrt_oracle_ray_valid.argtypes = [C.c_void_p, C.c_void_p]
    lib.tcrt_oracle_trace_rays.restype = C.c_int
    lib.tcrt_oracle_trace_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                           C.POINTER(C.c_ulonglong), C.POINTER(O.OracleCounters)]
    lib.tcrt_oracle_intersect_rays.restype = C.c_int
    lib.tcrt_oracle_intersect_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_ulonglong)]
    return lib


def _c(a):
    return np.ascontiguousarray(a, F32)


def oracle_trace(lib, flat, p, origins, dirs):
    """(rgb (n, 3), n_invalid, counters dict) of the oracle."""
    o, d = _c(origins), _c(dirs)
    n = d.shape[0]
    rgb = np.empty((n, 3), F32)
    bad = C.c_ulonglong()
    cnt = O.OracleCounters()
    assert lib.tcrt_oracle_trace_rays(C.byref(flat), C.byref(p), n, o.ctypes.data, int(o.shape == (3,)), d.ctypes.data,
                                      rgb.ctypes.data, C.byref(bad), C.byref(cnt)) == 0
    return rgb, int(bad.value), cnt.as_dict()


def oracle_hits(lib, flat, p, origins, dirs):
    o, d = _c(origins), _c(dirs)
    n = d.shape[0]
    out = {"object": np.empty(n, np.int32), "distance": np.empty(n, F32), "normal": np.empty((n, 3), F32)}
    bad = C.c_ulonglong()
    assert lib.tcrt_oracle_intersect_rays(C.byref(flat), C.byref(p), n, o.ctypes.data, int(o.shape == (3,)), d.ctypes.data,
                                          *(out[k].ctypes.data for k in HIT_NAMES), C.byref(bad)) == 0
    return out, int(bad.value)


def valid_rule(origins, dirs):
    """The validity rule of tcrt.h in numpy float32."""
    o = np.broadcast_to(_c(origins), _c(dirs).shape)
    d = _c(dirs)
    with np.errstate(all="ignore"):
        s = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
        return (np.isfinite(o).all(1) & np.isfinite(d).all(1) & (np.abs(o) <= F32(2.0 ** 40)).all(1)
                & (np.abs(s - F32(1)) <= F32(2.0 ** -21)))


def eye_rays(cam, w, h, order="x"):
    """The frame's primary rays (Camera::createEyeRay at x / W, z / H): origin = eye, direction = normalize(pixel - eye)
    in float32.  order "x": x-major like frames (ray x*H + z); "tile": the band kernel's 4x8-tile claim order; "shuffle": a
    fixed permutation.  Returns (origins (n, 3), directions (n, 3), pixel index x*H + z of each ray)."""
    x, z = np.meshgrid(np.arange(w), np.arange(h), indexing="ij")
    x, z = x.ravel(), z.ravel()
    if order == "tile":
        assert w % 4 == 0 and h % 8 == 0
        t, i = np.divmod(np.arange(w * h), 32)
        tx, tz = np.divmod(t, h // 8)
        x, z = tx * 4 + i % 4, tz * 8 + i // 4
    elif order == "shuffle":
        perm = np.random.default_rng(7).permutation(w * h)
        x, z = x[perm], z[perm]
    dx = x.astype(F32) / F32(w)
    dy = z.astype(F32) / F32(h)
    sx = dx * F32(cam.screen_width) - F32(cam.screen_halfwidth)
    sy = dy * F32(cam.screen_height) - F32(cam.screen_halfheight)
    so, hz, vt = (np.array(v[:], F32) for v in (cam.screen_origin, cam.horizontal, cam.vertical))
    pixel = so + hz * sx[:, None]
    pixel = pixel + vt * sy[:, None]
    eye = np.array(cam.eye[:], F32)
    dirs = api.normalize_like_reference(pixel - eye)
    return np.ascontiguousarray(np.broadcast_to(eye, dirs.shape)), np.ascontiguousarray(dirs), x * h + z


def assert_hits_equal(got, want, what=""):
    for k in HIT_NAMES:
        if k not in got:
            continue
        g, w = np.ascontiguousarray(got[k]).view(np.uint32), np.ascontiguousarray(want[k]).view(np.uint32)
        assert g.shape == w.shape, f"{what} {k}: shape {g.shape} vs {w.shape}"
        bad = int((g != w).reshape(len(g), int(np.prod(g.shape[1:]))).any(-1).sum())
        assert bad == 0, f"{what} {k}: {bad} of {len(g)} rays differ bitwise"


def _counters(st):
    return st.rays_primary, st.rays_shadow, st.rays_reflect


def _want_counters(cnt):
    return cnt["rays_primary"], cnt["rays_shadow"], cnt["rays_reflect"]


# ---- no device needed ------------------------------------------------------------------------------------------------

def test_ray_entry_points_are_exported():
    lib = _ffi.load()
    for name in ENTRY_POINTS:
        assert hasattr(lib, name), name


def test_ray_entry_points_refuse_a_null_context():
    lib = _ffi.load()
    p = api.default_params(8, 8, 2)
    o = np.zeros((4, 3), F32)
    d = np.tile(np.array([1, 0, 0], F32), (4, 1))
    rgb = np.full((4, 3), 7.0, F32)
    obj = np.full(4, 7, np.int32)
    bad = C.c_ulonglong(99)
    st = _ffi.TcrtStats()
    io = (o.ctypes.data_as(C.c_void_p), 0, d.ctypes.data_as(C.c_void_p))
    assert lib.tcrt_trace_rays(None, C.byref(p), 4, *io, rgb.ctypes.data_as(C.c_void_p), C.byref(bad), C.byref(st)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_trace_rays(None, None, 0, None, 0, None, None, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_intersect_rays(None, C.byref(p), 4, *io, obj.ctypes.data_as(C.c_void_p), None, None, C.byref(bad),
                                   C.byref(st)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_intersect_rays(None, C.byref(p), 1 << 62, *io, obj.ctypes.data_as(C.c_void_p), None, None, None,
                                   None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_trace_rays_device(None, 0, C.byref(p), 4, *io, rgb.ctypes.data_as(C.c_void_p), None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_intersect_rays_device(None, -1, C.byref(p), 4, *io, None, None, None, None, None) == _ffi.TCRT_ERR_INVALID
    assert bad.value == 99 and (rgb == 7.0).all() and (obj == 7).all()


def test_without_a_device_there_is_no_context():
    if api.device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(api.TcrtError) as e:
        api.Context([0])
    assert e.value.code == _ffi.TCRT_ERR_NO_DEVICE


@pytest.mark.parametrize("key", ["default_96x54_d5", "two_mirrors_64x48_d50", "synth256_96x80_d10", "boxes_3_14_96x80_d12"])
def test_oracle_rays_reproduce_golden_and_oracle_frames(rays_lib, hits_oracle, golden, golden_frames, key):
    """The eye rays of a frame, built in numpy, traced by oracle_rays.c: the reference's own golden frame and the oracle's
    render, ray counters included, and the oracle's primary hits."""
    m = golden["frames"][key]
    scene, cam = make_scene(m["scene"])
    flat, c = scene.flatten(), cam.export()
    p = api.default_params(m["W"], m["H"], m["depth"])
    o, d, pix = eye_rays(c, p.width, p.height)
    assert (pix == np.arange(p.width * p.height)).all()
    want, cnt = O.render(flat, c, p)
    for origins in (o, o[0].copy()):
        rgb, n_bad, got_cnt = oracle_trace(rays_lib, flat, p, origins, d)
        assert n_bad == 0
        assert_bit_identical(rgb.reshape(want.shape), golden_frames[key], f"{key} golden")
        assert _want_counters(got_cnt) == _want_counters(cnt)
    from test_hit_buffers import primary_hits
    ph = primary_hits(hits_oracle, flat, c, p)
    got, n_bad = oracle_hits(rays_lib, flat, p, o, d)
    assert n_bad == 0
    assert_hits_equal(got, {k: v.reshape(got[k].shape) for k, v in ph.items()}, key)


@pytest.fixture(scope="module")
def hits_oracle(tmp_path_factory):
    """tests/oracle_hits.c: the primary hits of a frame, for the eye-ray check above."""
    so = tmp_path_factory.mktemp("oracle_hits") / "liboracle_hits.so"
    subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", os.path.join(ROOT, "tests", "oracle_hits.c"),
                    "-o", str(so), "-lm"], check=True)
    lib = C.CDLL(str(so))
    lib.tcrt_oracle_primary_hits.restype = C.c_int
    lib.tcrt_oracle_primary_hits.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                             C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


def test_oracle_rays_on_a_lattice_equal_the_oracle_render(rays_lib):
    scene, cam = make_scene("lattice:1:4")
    flat, c = scene.flatten(), cam.export()
    p = api.default_params(64, 48, 8)
    o, d, _ = eye_rays(c, 64, 48, "shuffle")
    want, cnt = O.render(flat, c, p)
    rgb, _, got_cnt = oracle_trace(rays_lib, flat, p, o, d)
    _, _, pix = eye_rays(c, 64, 48, "shuffle")
    assert_bit_identical(rgb, want.reshape(-1, 3)[pix], "lattice, shuffled eye rays")
    assert _want_counters(got_cnt) == _want_counters(cnt)


def test_normalized_directions_are_valid():
    """normalize_like_reference of 2^20 vectors scaled by 2^-60 .. 2^60 (squared lengths normal floats): all valid."""
    rng = np.random.default_rng(1)
    v = rng.standard_normal((1 << 20, 3)).astype(F32)
    v *= np.exp2(rng.uniform(-60, 60, (len(v), 1))).astype(F32)
    v = v[np.isfinite(((v.astype(np.float64)) ** 2).sum(1))]
    d = api.normalize_like_reference(v)
    assert len(d) >= 1_000_000
    assert valid_rule(np.zeros(3, F32), d).all()
    s = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    assert np.abs(s.astype(np.float64) - 1).max() <= 6 * 2.0 ** -24


def normalize_in_c(v):
    """The same normalisation through the oracle's v3_normalize (via its primary ray): a check on the numpy restatement."""
    lib = O.lib()
    p = api.default_params(1, 1, 0)
    cam = api.Camera().export()
    out = []
    for x in v:
        # screen point = eye + x: one pixel whose screen origin is moved there
        for k in range(3):
            cam.screen_origin[k] = cam.eye[k] + float(x[k])
        cam.screen_halfwidth = cam.screen_halfheight = 0.0
        o3, d3 = (C.c_float * 3)(), (C.c_float * 3)()
        assert lib.tcrt_oracle_primary_ray(C.byref(cam), C.byref(p), 0, 0, o3, d3) == 0
        out.append(list(d3))
    return np.array(out, F32)


def test_normalize_like_reference_is_the_oracles_normalize():
    rng = np.random.default_rng(2)
    eye = np.array(api.Camera().export().eye[:], F32)
    v = rng.uniform(-3, 3, (200, 3)).astype(F32)
    v = (eye + v) - eye                                # exactly representable differences
    assert np.array_equal(bits(normalize_in_c(v)), bits(api.normalize_like_reference(v)))


def _find(target_s, lo, hi):
    """A direction (x, y, 0) whose s is exactly target_s (float32): x near 1, y scanned."""
    xs = np.nextafter(F32(lo), F32(2)) + np.arange(-64, 64, dtype=F32) * np.spacing(F32(lo))
    ys = np.linspace(0, hi, 1 << 16, dtype=F32)
    for x in xs:
        s = (x * x + ys * ys) + F32(0) * F32(0)
        k = np.nonzero(s == F32(target_s))[0]
        if len(k):
            return np.array([x, ys[k[0]], 0], F32)
    raise AssertionError(f"no direction with s = {target_s!r}")


def boundary_directions():
    """(accepted, refused): s = 1 + 2^-21 and 1 - 2^-21, and their float neighbours one ulp outside."""
    up, dn = F32(1 + 2.0 ** -21), F32(1 - 2.0 ** -21)
    up_out, dn_out = np.nextafter(up, F32(2)), np.nextafter(dn, F32(0))
    acc = [_find(up, 1.0, 2e-3), _find(dn, 1 - 2.0 ** -22, 2e-3)]
    ref = [_find(up_out, 1.0, 2e-3), _find(dn_out, 1 - 2.0 ** -22, 2e-3)]
    return np.array(acc), np.array(ref)


def crafted_rays():
    """(origins, directions, valid) covering every clause of the validity rule."""
    acc, ref = boundary_directions()
    e = np.array([0.0, 0.0, 1.0], F32)
    big = F32(2.0 ** 40)
    nan, inf = F32(np.nan), F32(np.inf)
    rows = [((0, 0, 0), acc[0], True), ((0, 0, 0), acc[1], True), ((0, 0, 0), ref[0], False), ((0, 0, 0), ref[1], False),
            ((0, 0, 0), (nan, 0, 1), False), ((0, 0, 0), (0, inf, 0), False), ((0, 0, 0), (0, 0, -inf), False),
            ((0, 0, 0), (0, 0, 0), False), ((nan, 0, 0), e, False), ((0, -inf, 0), e, False),
            ((big, -big, big), e, True), ((np.nextafter(big, F32(np.inf)), 0, 0), e, False),
            ((0, 0, -np.nextafter(big, F32(np.inf))), e, False), ((0, 0, 0), (1, 0, 0), True), ((0, 0, 0), (0, -1, 0), True)]
    o = np.array([r[0] for r in rows], F32)
    d = np.array([r[1] for r in rows], F32)
    return o, d, np.array([r[2] for r in rows])


def test_validity_rule_at_its_boundaries(rays_lib):
    o, d, want = crafted_rays()
    s = (d[:, 0] * d[:, 0] + d[:, 1] * d[:, 1]) + d[:, 2] * d[:, 2]
    assert s[0] == F32(1 + 2.0 ** -21) and s[1] == F32(1 - 2.0 ** -21)
    assert s[2] == np.nextafter(s[0], F32(2)) and s[3] == np.nextafter(s[1], F32(0))
    assert (valid_rule(o, d) == want).all()
    assert [rays_lib.tcrt_oracle_ray_valid(o[i].ctypes.data, d[i].ctypes.data) for i in range(len(o))] == list(want.astype(int))


def test_oracle_marks_invalid_rays(rays_lib):
    scene, cam = make_scene("default")
    flat = scene.flatten()
    p = api.default_params(1, 1, 5)
    o, d, valid = crafted_rays()
    o = o + np.array(cam.export().eye[:], F32) * valid[:, None]   # the valid rays start at the eye
    rgb, n_bad, cnt = oracle_trace(rays_lib, flat, p, o, d)
    assert n_bad == int((~valid).sum()) and cnt["rays_primary"] == int(valid.sum())
    assert (rgb[~valid].view(np.uint32) == 0x7fc00000).all()
    assert np.isfinite(rgb[valid]).all()
    hits, n_bad = oracle_hits(rays_lib, flat, p, o, d)
    assert n_bad == int((~valid).sum())
    assert (hits["object"][~valid] == -2).all() and (hits["distance"][~valid].view(np.uint32) == 0x7fc00000).all()
    assert (hits["normal"][~valid].view(np.uint32) == 0x7fc00000).all() and (hits["object"][valid] >= -1).all()


# ---- on the GPU ------------------------------------------------------------------------------------------------------

def _upload_spec(ctx, spec):
    if spec == "inside_sphere":
        from test_adaptive_frames import _inside_sphere_scene
        s, c = _inside_sphere_scene()
    elif spec == "far_camera":
        s, cam = make_scene("synth256")
        c = cam.export()
        for k, delta in enumerate((600.0, -450.0, 300.0)):
            c.eye[k] += delta
            c.screen_origin[k] += delta
    else:
        s, cam = make_scene(spec)
        c = cam.export()
    flat = s.flatten()
    ctx.upload_flat(flat, c)
    return s, flat, c


def check_eye_rays(ctx, c, p, what, hits=True):
    """Eye rays of the frame p (x-major; per-ray and shared origin) traced as a batch equal tcrt_render, counters included;
    intersect_rays equals tcrt_hit_buffers."""
    frame, st = ctx.render(p)
    frame = frame.copy()
    o, d, _ = eye_rays(c, p.width, p.height)
    for origins in (o, o[0].copy()):
        rgb, n_bad, st_r = ctx.trace_rays(p, origins, d)
        assert n_bad == 0, what
        assert_bit_identical(rgb.reshape(frame.shape), frame, what)
        assert _counters(st_r) == _counters(st), what
    if hits:
        want, _ = ctx.hit_buffers(p)
        got, n_bad, _ = ctx.intersect_rays(p, o, d)
        assert n_bad == 0
        assert_hits_equal(got, {k: v.reshape(got[k].shape) for k, v in want.items()}, what)


@gpu
def test_eye_rays_reproduce_every_dispatch_class(gpu_ctx):
    from test_kernel_variants import DEPTHS, NAMES, _upload
    for name in NAMES:
        s, flat, c = _upload(gpu_ctx, name)
        for depth in DEPTHS:
            w, h = (40, 32) if depth > 64 else (48, 40)
            check_eye_rays(gpu_ctx, c, api.default_params(w, h, depth), f"{name} d{depth}", hits=depth == 0)


@gpu
@pytest.mark.parametrize("spec,w,h,d", [("default", 160, 120, 50), ("two_mirrors", 96, 80, 50), ("synth256", 160, 128, 10),
                                        ("lattice:1:4", 128, 96, 8), ("inside_sphere", 96, 72, 8), ("far_camera", 96, 72, 8)])
def test_eye_rays_reproduce_named_scenes(gpu_ctx, spec, w, h, d):
    s, flat, c = _upload_spec(gpu_ctx, spec)
    if spec in ("synth256", "inside_sphere"):
        assert gpu_ctx.scene_structures()["grid_cells"] > 0
    check_eye_rays(gpu_ctx, c, api.default_params(w, h, d), spec)


def arbitrary_rays(ctx, flat, c, spec, rng):
    """Every kind of ray the batch must take: random origins in the scene's box, surface points from the hit buffers (at
    0 and 1e-3 along the normal, grazing directions), origins inside spheres, far origins, directions with zero
    components, rays aimed at lights, and an equirectangular panorama from the eye."""
    n_s = flat.n_spheres
    sph = np.ctypeslib.as_array(flat.sphere_geom, (n_s * 4,)).reshape(n_s, 4) if n_s else np.zeros((0, 4), F32)
    info = np.ctypeslib.as_array(flat.obj_info, (flat.n_objects * 4,)).reshape(-1, 4)
    org = np.ctypeslib.as_array(flat.obj_origin, (flat.n_objects * 4,)).reshape(-1, 4)[:, :3]
    lights = org[info[:, 2] != 0]
    eye = np.array(c.eye[:], F32)
    lo = np.minimum(sph[:, :3].min(0) if n_s else eye, eye) - 2
    hi = np.maximum(sph[:, :3].max(0) if n_s else eye, eye) + 2
    parts = []
    def rnd_dir(n):
        return api.normalize_like_reference(rng.standard_normal((n, 3)).astype(F32))
    n = 4096
    parts.append((rng.uniform(lo, hi, (n, 3)).astype(F32), rnd_dir(n)))
    # surface points: the hits of the frame's eye rays
    p = api.default_params(64, 48, 0)
    hb, _ = ctx.hit_buffers(p)
    o_e, d_e, _ = eye_rays(c, 64, 48)
    hitm = hb["object"].ravel() >= 0
    t = hb["distance"].ravel()[hitm]
    P = (d_e[hitm] * t[:, None]) + o_e[hitm]
    N = hb["normal"].reshape(-1, 3)[hitm]
    for off in (F32(0), F32(1e-3)):
        Q = P + N * off
        graze = api.normalize_like_reference(np.cross(N, rnd_dir(len(N))) + N * F32(1e-3))
        parts.append((Q, graze))
        parts.append((Q, rnd_dir(len(Q))))
    if n_s:
        k = rng.integers(0, n_s, 1024)
        parts.append((sph[k, :3] + rng.uniform(-.3, .3, (1024, 3)).astype(F32) * np.sqrt(sph[k, 3:4]), rnd_dir(1024)))
        target = sph[rng.integers(0, n_s, 3 * 512), :3]
    else:
        target = np.zeros((3 * 512, 3), F32)
    for i, r in enumerate((600.0, 1e6, 2.0 ** 40)):
        far = api.normalize_like_reference(rng.standard_normal((512, 3)).astype(F32)) * F32(r)
        far = np.clip(far, -F32(2.0 ** 40), F32(2.0 ** 40))
        parts.append((far, api.normalize_like_reference(target[512 * i:512 * (i + 1)] - far)))
    axis = np.array([(1, 0, 0), (-1, 0, 0), (0, 1, 0), (0, -1, 0), (0, 0, 1), (0, 0, -1), (1, 1, 0), (0, -1, 1), (1, 0, -1)], F32)
    parts.append((rng.uniform(lo, hi, (len(axis) * 64, 3)).astype(F32), api.normalize_like_reference(np.repeat(axis, 64, 0))))
    if len(lights):
        src = rng.uniform(lo, hi, (256 * len(lights), 3)).astype(F32)
        parts.append((src, api.normalize_like_reference(np.repeat(lights, 256, 0) - src)))
    th, ph = np.meshgrid(np.linspace(0, 2 * np.pi, 96, endpoint=False), np.linspace(-np.pi / 2, np.pi / 2, 48), indexing="ij")
    pano = np.stack([np.cos(ph) * np.cos(th), np.cos(ph) * np.sin(th), np.sin(ph)], -1).reshape(-1, 3).astype(F32)
    parts.append((np.broadcast_to(eye, pano.shape), api.normalize_like_reference(pano)))
    o = np.ascontiguousarray(np.concatenate([a for a, _ in parts]), F32)
    d = np.ascontiguousarray(np.concatenate([b for _, b in parts]), F32)
    keep = valid_rule(o, d)
    return o[keep], d[keep], (eye, api.normalize_like_reference(pano))


ARB_SCENES = ["default", "two_mirrors", "synth256", "boxes:3:14", "inside_sphere"]


@gpu
@pytest.mark.parametrize("spec", ARB_SCENES)
def test_arbitrary_rays_match_the_oracle(gpu_ctx, rays_lib, spec):
    rng = np.random.default_rng(hash(spec) % 1000)
    s, flat, c = _upload_spec(gpu_ctx, spec)
    o, d, (eye, pano) = arbitrary_rays(gpu_ctx, flat, c, spec, rng)
    assert len(o) > 5000
    settings = [dict(depth=0), dict(depth=1), dict(depth=5), dict(depth=50), dict(depth=5, shadows=False),
                dict(depth=5, reflections=False), dict(depth=50, null=(0.1, -0.0, 2.5), far=40.0)]
    for kw in settings:
        p = api.default_params(1, 1, kw["depth"], shadows=kw.get("shadows", True), reflections=kw.get("reflections", True))
        if "null" in kw:
            for k in range(3):
                p.null_color[k] = kw["null"][k]
            p.far_dist = kw["far"]
        what = f"{spec} {kw}"
        want, n_bad, cnt = oracle_trace(rays_lib, flat, p, o, d)
        got, g_bad, st = gpu_ctx.trace_rays(p, o, d)
        assert n_bad == g_bad == 0, what
        assert_bit_identical(got, want, what)
        assert _counters(st) == _want_counters(cnt), what
        if kw["depth"] in (0, 50):
            want_h, _ = oracle_hits(rays_lib, flat, p, o, d)
            got_h, _, _ = gpu_ctx.intersect_rays(p, o, d)
            assert_hits_equal(got_h, want_h, what)
    # the shared-origin panorama
    p = api.default_params(1, 1, 10)
    want, _, cnt = oracle_trace(rays_lib, flat, p, eye, pano)
    got, _, st = gpu_ctx.trace_rays(p, eye, pano)
    assert_bit_identical(got, want, f"{spec} panorama")
    assert _counters(st) == _want_counters(cnt)


@gpu
def test_invalid_rays_in_a_batch(gpu_ctx, rays_lib):
    s, flat, c = _upload_spec(gpu_ctx, "synth256")
    p = api.default_params(1, 1, 10)
    rng = np.random.default_rng(5)
    o_v, d_v, _ = eye_rays(c, 64, 48)
    o_x, d_x, valid_x = crafted_rays()
    bad = ~valid_x
    n = len(o_v) + 3 * int(bad.sum())
    pos = np.sort(rng.choice(n, 3 * int(bad.sum()), replace=False))
    is_bad = np.zeros(n, bool)
    is_bad[pos] = True
    o = np.empty((n, 3), F32)
    d = np.empty((n, 3), F32)
    o[~is_bad], d[~is_bad] = o_v, d_v
    o[is_bad], d[is_bad] = np.tile(o_x[bad], (3, 1)), np.tile(d_x[bad], (3, 1))
    clean, _, st_c = gpu_ctx.trace_rays(p, o_v, d_v)
    clean = clean.copy()
    for grid in (True, False):
        if not grid:
            s, flat, c = _upload_spec(gpu_ctx, "default")
            o_v2, d_v2, _ = eye_rays(c, 64, 48)
            o[~is_bad], d[~is_bad] = o_v2, d_v2
            clean, _, st_c = gpu_ctx.trace_rays(p, o_v2, d_v2)
            clean = clean.copy()
        got, n_bad, st = gpu_ctx.trace_rays(p, o, d)
        assert n_bad == int(is_bad.sum()) and st.rays_primary == int((~is_bad).sum())
        assert (got[is_bad].view(np.uint32) == 0x7fc00000).all()
        assert_bit_identical(got[~is_bad], clean, "valid rays among invalid ones")
        assert _counters(st) == _counters(st_c)
        want, w_bad, _ = oracle_trace(rays_lib, flat, p, o, d)
        assert w_bad == n_bad
        assert_bit_identical(got, want, "mixed batch against the oracle")
        h, h_bad, st_h = gpu_ctx.intersect_rays(p, o, d)
        want_h, _ = oracle_hits(rays_lib, flat, p, o, d)
        assert h_bad == n_bad and st_h.rays_primary == int((~is_bad).sum())
        assert_hits_equal(h, want_h, "mixed batch hits")
    # all invalid
    got, n_bad, st = gpu_ctx.trace_rays(p, o_x[bad], d_x[bad])
    assert n_bad == int(bad.sum()) and st.rays_primary == 0 and (got.view(np.uint32) == 0x7fc00000).all()
    h, n_bad, _ = gpu_ctx.intersect_rays(p, o_x[bad], d_x[bad])
    assert n_bad == int(bad.sum()) and (h["object"] == -2).all()


@gpu
def test_validity_boundaries_on_the_gpu(gpu_ctx):
    _upload_spec(gpu_ctx, "default")
    o, d, valid = crafted_rays()
    got, n_bad, _ = gpu_ctx.trace_rays(api.default_params(1, 1, 3), o, d)
    assert n_bad == int((~valid).sum())
    assert ((got.view(np.uint32) == 0x7fc00000).all(1) == ~valid).all()
    assert np.isfinite(got[valid]).all()


@gpu
@pytest.mark.parametrize("n", [0, 1, 31, 33])
def test_small_batches(gpu_ctx, rays_lib, n):
    s, flat, c = _upload_spec(gpu_ctx, "two_mirrors")
    p = api.default_params(1, 1, 20)
    o, d, _ = eye_rays(c, 16, 8, "shuffle")
    o, d = o[:n], d[:n]
    got, n_bad, st = gpu_ctx.trace_rays(p, o, d)
    want, _, cnt = oracle_trace(rays_lib, flat, p, o, d)
    assert_bit_identical(got.reshape(n, 1, 3), want.reshape(n, 1, 3), f"n = {n}")
    assert _counters(st) == _want_counters(cnt) and st.gpu_launches == (1 if n else 0)
    h, _, st = gpu_ctx.intersect_rays(p, o, d)
    assert_hits_equal(h, oracle_hits(rays_lib, flat, p, o, d)[0], f"n = {n}")


@gpu
def test_a_batch_of_several_pieces_is_the_4k_frame(gpu_ctx):
    """The 4K eye rays (8.3 M: two pieces), and the same rays followed by their first half again (12.4 M: three pieces on
    three render streams), against the 4K frame, at the piece boundaries and everywhere."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    p = api.default_params(3840, 2160, 5)
    frame, st = gpu_ctx.render(p)
    frame = frame.reshape(-1, 3).copy()
    o, d, _ = eye_rays(c, 3840, 2160)
    m = len(o)
    for k, (oo, dd) in enumerate(((o, d), (np.concatenate([o, o[:m // 2]]), np.concatenate([d, d[:m // 2]])))):
        want = frame if k == 0 else np.concatenate([frame, frame[:m // 2]])
        rgb, n_bad, st_r = gpu_ctx.trace_rays(p, oo, dd)
        assert n_bad == 0 and st_r.gpu_launches == (len(oo) + PIECE - 1) // PIECE == 2 + k
        for b in range(PIECE, len(oo), PIECE):
            assert_bit_identical(rgb[b - 64:b + 64].reshape(-1, 1, 3), want[b - 64:b + 64].reshape(-1, 1, 3), f"piece boundary {b}")
        assert_bit_identical(rgb.reshape(-1, 1, 3), want.reshape(-1, 1, 3), f"{len(oo)} eye rays")
        if k == 0:
            assert _counters(st_r) == _counters(st)


GUARD = 64


@gpu
def test_destinations(gpu_ctx):
    """Pinned and pageable inputs and outputs (with guard words), every non-empty subset of hit outputs, and the device forms
    with torch tensors: identical bits."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    p = api.default_params(1, 1, 8)
    o, d, _ = eye_rays(c, 1024, 768, "tile")          # 786 K rays: the staged copy-out of pageable outputs
    n = len(o)
    ref, _, st_ref = gpu_ctx.trace_rays(p, o, d)
    ref = ref.copy()
    ref_h, _, _ = gpu_ctx.intersect_rays(p, o, d)
    ref_h = {k: v.copy() for k, v in ref_h.items()}
    bufs = []
    def pinned(shape, dtype):
        hb = api.HostBuffer(int(np.prod(shape)) * np.dtype(dtype).itemsize + 2 * GUARD * 4)
        bufs.append(hb)
        a = hb.array(np.uint32, (hb.nbytes // 4,))
        a[:] = 0xDEADBEEF
        return a[GUARD:GUARD + int(np.prod(shape)) * np.dtype(dtype).itemsize // 4].view(dtype).reshape(shape), a
    def pageable(shape, dtype):
        a = np.full(int(np.prod(shape)) * np.dtype(dtype).itemsize // 4 + 2 * GUARD, 0xDEADBEEF, np.uint32)
        return a[GUARD:len(a) - GUARD].view(dtype).reshape(shape), a
    for in_kind in (pinned, pageable):
        oi, _ = in_kind((n, 3), F32)
        di, _ = in_kind((n, 3), F32)
        oi[:], di[:] = o, d
        for out_kind in (pinned, pageable):
            rgb, whole = out_kind((n, 3), F32)
            got, _, st = gpu_ctx.trace_rays(p, oi, di, out=rgb)
            assert_bit_identical(got.reshape(-1, 1, 3), ref.reshape(-1, 1, 3), f"{in_kind.__name__} -> {out_kind.__name__}")
            assert (whole[:GUARD] == 0xDEADBEEF).all() and (whole[-GUARD:] == 0xDEADBEEF).all()
            assert _counters(st) == _counters(st_ref)
            for mask in range(1, 8):
                out, wholes = {}, []
                for b, (name, dtype, tail) in enumerate(api.Context.HIT_BUFFERS):
                    if mask >> b & 1:
                        out[name], w = out_kind((n,) + tail, dtype)
                        wholes.append(w)
                got_h, _, _ = gpu_ctx.intersect_rays(p, oi, di, out=out)
                assert set(got_h) == set(out)
                assert_hits_equal(got_h, ref_h, f"hit subset {mask}")
                for w in wholes:
                    assert (w[:GUARD] == 0xDEADBEEF).all() and (w[-GUARD:] == 0xDEADBEEF).all()
    import torch
    dev = torch.device("cuda:0")
    to, td = torch.from_numpy(o).to(dev), torch.from_numpy(d).to(dev)
    trgb = torch.full((n, 3), 7.0, device=dev)
    torch.cuda.synchronize()
    n_bad, st = gpu_ctx.trace_rays_device(p, n, to.data_ptr(), td.data_ptr(), trgb.data_ptr())
    assert n_bad == 0 and _counters(st) == _counters(st_ref)
    assert_bit_identical(trgb.cpu().numpy().reshape(-1, 1, 3), ref.reshape(-1, 1, 3), "device form")
    tshared = torch.from_numpy(o[0].copy()).to(dev)
    torch.cuda.synchronize()
    gpu_ctx.trace_rays_device(p, n, tshared.data_ptr(), td.data_ptr(), trgb.data_ptr(), shared_origin=True)
    assert_bit_identical(trgb.cpu().numpy().reshape(-1, 1, 3), ref.reshape(-1, 1, 3), "device form, shared origin")
    tobj = torch.full((n,), 7, dtype=torch.int32, device=dev)
    tdist = torch.zeros(n, device=dev)
    tnorm = torch.zeros((n, 3), device=dev)
    torch.cuda.synchronize()
    gpu_ctx.intersect_rays_device(p, n, to.data_ptr(), td.data_ptr(), tobj.data_ptr(), tdist.data_ptr(), tnorm.data_ptr())
    assert_hits_equal({"object": tobj.cpu().numpy(), "distance": tdist.cpu().numpy(), "normal": tnorm.cpu().numpy()}, ref_h,
                      "device form hits")
    gpu_ctx.intersect_rays_device(p, n, to.data_ptr(), td.data_ptr(), distance=tdist.data_ptr())
    assert_hits_equal({"distance": tdist.cpu().numpy()}, ref_h, "device form, distance only")
    # a wrong slot, a host pointer
    with pytest.raises(api.TcrtError) as e:
        gpu_ctx.trace_rays_device(p, n, to.data_ptr(), td.data_ptr(), trgb.data_ptr(), slot=1)
    assert e.value.code == _ffi.TCRT_ERR_INVALID
    with pytest.raises(api.TcrtError) as e:
        gpu_ctx.trace_rays_device(p, n, o.ctypes.data, td.data_ptr(), trgb.data_ptr())
    assert e.value.code == _ffi.TCRT_ERR_INVALID


@gpu
def test_error_codes(gpu_ctx):
    lib = _ffi.load()
    o = np.zeros((4, 3), F32)
    d = np.tile(np.array([1, 0, 0], F32), (4, 1))
    rgb = np.empty((4, 3), F32)
    fresh = api.Context([0])
    with pytest.raises(api.TcrtError) as e:
        fresh.trace_rays(api.default_params(1, 1, 2), o, d)
    assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
    fresh.close()
    _upload_spec(gpu_ctx, "default")
    p = api.default_params(1, 1, 2)
    h = gpu_ctx._h
    io = (o.ctypes.data_as(C.c_void_p), 0, d.ctypes.data_as(C.c_void_p))
    r = rgb.ctypes.data_as(C.c_void_p)
    assert lib.tcrt_trace_rays(h, C.byref(p), 4, *io, None, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_trace_rays(h, C.byref(p), 4, None, 0, io[2], r, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_trace_rays(h, C.byref(p), 1 << 62, *io, r, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_intersect_rays(h, C.byref(p), 4, *io, None, None, None, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_trace_rays(h, None, 4, *io, r, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_trace_rays(h, C.byref(p), 0, None, 0, None, r, None, None) == _ffi.TCRT_OK
    p.max_depth = 255
    assert lib.tcrt_trace_rays(h, C.byref(p), 4, *io, r, None, None) == _ffi.TCRT_ERR_UNSUPPORTED
    p.max_depth = -1
    assert lib.tcrt_trace_rays(h, C.byref(p), 4, *io, r, None, None) == _ffi.TCRT_ERR_INVALID


@gpu
def test_batches_leave_the_last_render_and_the_camera_alone(gpu_ctx, tmp_path):
    scene, cam = make_scene("two_mirrors")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    p = api.default_params(64, 48, 20)
    frame, _ = gpu_ctx.render(p)
    frame = frame.copy()
    gpu_ctx.write_txt(p, str(tmp_path / "a.txt"))
    gpu_ctx.write_ppm(p, str(tmp_path / "a.ppm"))
    o, d, _ = eye_rays(c, 64, 48)
    ref, _, _ = gpu_ctx.trace_rays(p, o, d)
    ref = ref.copy()
    # two frames in flight around a batch
    buf = [api.HostBuffer(64 * 48 * 12) for _ in range(2)]
    outs = [b.array(F32, (64, 48, 3)) for b in buf]
    t = [gpu_ctx.render_async(p, 0, 64, outs[k]) for k in range(2)]
    got, _, _ = gpu_ctx.trace_rays(p, o, d)
    assert_bit_identical(got.reshape(-1, 1, 3), ref.reshape(-1, 1, 3), "with two frames in flight")
    h, _, _ = gpu_ctx.intersect_rays(p, o, d)
    for k in range(2):
        gpu_ctx.wait(t[k])
        assert_bit_identical(outs[k], frame, "frame in flight")
    assert_bit_identical(gpu_ctx.download(np.empty_like(frame)), frame, "last render")
    gpu_ctx.write_txt(p, str(tmp_path / "b.txt"))
    gpu_ctx.write_ppm(p, str(tmp_path / "b.ppm"))
    assert (tmp_path / "a.txt").read_bytes() == (tmp_path / "b.txt").read_bytes()
    assert (tmp_path / "a.ppm").read_bytes() == (tmp_path / "b.ppm").read_bytes()
    # a new camera changes frames, not batches
    c2 = cam.export()
    for k in range(3):
        c2.eye[k] += 0.5
        c2.screen_origin[k] += 0.5
    gpu_ctx.set_camera(c2)
    got, _, _ = gpu_ctx.trace_rays(p, o, d)
    assert_bit_identical(got.reshape(-1, 1, 3), ref.reshape(-1, 1, 3), "after tcrt_set_camera")


@gpu
@pytest.mark.parametrize("n_bands", [2, 3])
def test_multi_device_batches(gpu_ctx, n_bands):
    n_dev = api.device_count()
    scene, cam = make_scene("synth256")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    p = api.default_params(1, 1, 10)
    o, d, _ = eye_rays(c, 320, 240, "tile")
    ref, _, st1 = gpu_ctx.trace_rays(p, o, d)
    ref = ref.copy()
    ref_h, _, _ = gpu_ctx.intersect_rays(p, o, d)
    ref_h = {k: v.copy() for k, v in ref_h.items()}
    multi = api.Context([i % n_dev for i in range(n_bands)])
    multi.upload(scene, cam)
    n = len(o)
    got, _, st = multi.trace_rays(p, o, d)
    assert_bit_identical(got.reshape(-1, 1, 3), ref.reshape(-1, 1, 3), f"{n_bands} devices")
    assert st.bands == [(n * i // n_bands, n * (i + 1) // n_bands) for i in range(n_bands)]
    assert _counters(st) == _counters(st1)
    h, _, st = multi.intersect_rays(p, o, d)
    assert_hits_equal(h, ref_h, f"{n_bands} devices hits")
    assert st.bands == [(n * i // n_bands, n * (i + 1) // n_bands) for i in range(n_bands)]
    multi.close()


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
    const int W = 96, H = 72;
    std::vector<Ray> rays;
    for (int x = 0; x < W; x++)
        for (int z = 0; z < H; z++) {
            Ray* r = camera.createEyeRay(((float)x) / W, ((float)z) / H);
            rays.push_back(*r);
            delete r;
        }
    GpuRayTracer rt;
    RenderSettings rs;
    rs.width = W; rs.height = H; rs.max_depth = 50;
    std::vector<float> rgb(rays.size() * 3), dist(rays.size()), normal(rays.size() * 3);
    std::vector<int> obj(rays.size());
    unsigned long long bad = 99;
    if (!rt.ok() || rt.setScene(scene, camera) || rt.traceRays(rs, rays, rgb.data(), &bad) ||
        rt.intersectRays(rs, rays, obj.data(), dist.data(), normal.data())) {
        fprintf(stderr, "%s\n", rt.lastError());
        return 1;
    }
    printf("%llu\n", bad);
    FILE* f = fopen("rays.bin", "wb");
    if (!f) return 1;
    fwrite(rgb.data(), 4, rgb.size(), f);
    fwrite(obj.data(), 4, obj.size(), f);
    fwrite(dist.data(), 4, dist.size(), f);
    fwrite(normal.data(), 4, normal.size(), f);
    return fclose(f) ? 1 : 0;
}
"""


@gpu
def test_cpp_trace_rays(gpu_ctx, tmp_path):
    src = tmp_path / "trace_rays.cpp"
    src.write_text(CPP_PROGRAM)
    libdir = os.path.join(ROOT, "tilecoderaytracer_b200")
    exe = tmp_path / "trace_rays"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), str(src),
                    "-L", libdir, "-ltcrt", f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert int(r.stdout.split()[-1]) == 0
    n = 96 * 72
    raw = np.fromfile(tmp_path / "rays.bin", dtype=np.uint32)
    rgb, obj, dist, normal = np.split(raw, [3 * n, 4 * n, 5 * n])
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    p = api.default_params(96, 72, 50)
    frame, _ = gpu_ctx.render(p)
    assert np.array_equal(rgb.view(F32).reshape(96, 72, 3).view(np.uint32), bits(frame)), "traceRays vs render"
    hb, _ = gpu_ctx.hit_buffers(p)
    assert np.array_equal(obj.view(np.int32), hb["object"].ravel())
    assert np.array_equal(dist, hb["distance"].ravel().view(np.uint32))
    assert np.array_equal(normal, hb["normal"].ravel().view(np.uint32))
