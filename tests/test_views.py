"""Multi-view frames (tcrt_render_views and its device form): one scene from a batch of cameras in one call, computed by the
render kernels' views mode.  View v must equal, bit for bit, the frame tcrt_render returns after tcrt_set_camera(cams[v]),
and the oracle's O.render(flat, cams[v], params); the ray counters must be the sums over the views.  Camera.aim builds
cameras with the reference's pose arithmetic."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import assert_bit_identical, bits, make_scene, quant8
from test_kernel_variants import DEPTHS, NAMES, _upload

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
PIECE = 1 << 22                 # pixels per piece at most (tcrt_api.cu kRayPiece)
F32 = np.float32
ENTRY_POINTS = ("tcrt_render_views", "tcrt_render_views_device", "tcrt_hcamera_aim")
# the literals of Camera::Camera() and Camera::setSceneTwoMirrors() (host_scene.cpp; Camera.cpp:22-38, 45-51)
DEFAULT_POSE = ((-4.0, -4.0, 1.5), (.1, -.08, 0.0), (.08, .1, .01))
TWO_MIRRORS_POSE = ((0.0, 0.0, 2.5), (1.0, -0.0, 0.0), (0.0, 1.0, -0.0))


def cam_bits(c):
    return np.frombuffer(bytes(c), np.uint32).copy()


def copy_cam(c):
    return _ffi.TcrtCamera.from_buffer_copy(bytes(c))


def moved(c, delta, fov=1.0):
    """c translated by delta, its screen scaled by fov (halfwidth = width / 2, as the reference sets it)."""
    m = copy_cam(c)
    for k in range(3):
        m.eye[k] += delta[k]
        m.screen_origin[k] += delta[k]
    m.screen_width = F32(c.screen_width * fov)
    m.screen_height = F32(c.screen_height * fov)
    m.screen_halfwidth = F32(m.screen_width / F32(2))
    m.screen_halfheight = F32(m.screen_height / F32(2))
    return m


def three_views(c):
    return [c, moved(c, (.3, -.2, .1)), moved(c, (-.25, .15, -.05), fov=.7)]


def aimed(so, horiz, outwards, screen=None):
    cam = api.Camera().aim(so, horiz, outwards)
    c = cam.export()
    if screen is not None:
        c.screen_width = c.screen_height = F32(screen)
        c.screen_halfwidth = c.screen_halfheight = F32(F32(screen) / F32(2))
    return c


def orbit_cameras(centre, radius, height, n):
    """n cameras on a circle around centre, each looking at it."""
    cams = []
    for k in range(n):
        a = 2 * math.pi * k / n
        so = (centre[0] + radius * math.cos(a), centre[1] + radius * math.sin(a), centre[2] + height)
        out = (centre[0] - so[0], centre[1] - so[1], centre[2] - so[2])
        horiz = (-math.sin(a), math.cos(a), 0.0)
        cams.append(aimed(so, horiz, out))
    return cams


def cube_cameras(p):
    """The six faces of a cube map at p: 2x2 screens one unit in front of the eye (90 degrees each)."""
    faces = [((1, 0, 0), (0, 1, 0)), ((-1, 0, 0), (0, -1, 0)), ((0, 1, 0), (-1, 0, 0)), ((0, -1, 0), (1, 0, 0)),
             ((0, 0, 1), (1, 0, 0)), ((0, 0, -1), (1, 0, 0))]
    return [aimed(tuple(p[k] + o[k] for k in range(3)), h, o, screen=2.0) for o, h in faces]


def _counters(st):
    return st.rays_primary, st.rays_shadow, st.rays_reflect


def per_view(ctx, p, cams):
    """What the views must equal: set_camera + render per view, and the summed counters."""
    frames, tot = [], np.zeros(3, np.int64)
    for c in cams:
        ctx.set_camera(c)
        img, st = ctx.render(p)
        frames.append(img.copy())
        tot += _counters(st)
    return np.stack(frames), tuple(int(t) for t in tot)


@pytest.fixture(scope="module")
def pair_ctx():
    """Two device slots (the same GPU when there is one): the second slot's columns start inside the stack, where a
    camera index taken from the launch-local column instead of the global one would show."""
    n_dev = api.device_count()
    ctx = api.Context([0, 1 % n_dev])
    yield ctx
    ctx.close()


def check_views(ctx, flat, p, cams, what, oracle=True, pair=None):
    """ctx.render_views against per-view set_camera + render, the oracle (small views) and, with `pair` (a two-slot context
    holding the same scene), the same call split over two slots."""
    got, st = ctx.render_views(p, cams)
    got = got.copy()
    want, cnt = per_view(ctx, p, cams)
    assert got.shape == (len(cams), p.width, p.height, 3)
    for v in range(len(cams)):
        assert_bit_identical(got[v], want[v], f"{what} view {v} vs set_camera + render")
    assert _counters(st) == cnt, what
    if pair is not None:
        got2, st2 = pair.render_views(p, cams)
        for v in range(len(cams)):
            assert_bit_identical(got2[v], want[v], f"{what} view {v} on two slots")
        assert _counters(st2) == cnt, what
    if oracle:
        tot = np.zeros(3, np.int64)
        for v, c in enumerate(cams):
            img, oc = O.render(flat, c, p)
            assert_bit_identical(got[v], img, f"{what} view {v} vs oracle")
            tot += (oc["rays_primary"], oc["rays_shadow"], oc["rays_reflect"])
        assert _counters(st) == tuple(int(t) for t in tot), what
    return got, st


# ---- without a GPU ---------------------------------------------------------------------------------------------------------

def test_view_entry_points_are_exported():
    lib = _ffi.load()
    for name in ENTRY_POINTS:
        assert hasattr(lib, name), name


def test_view_entry_points_refuse_a_null_context():
    lib = _ffi.load()
    p = api.default_params(4, 4, 2)
    cams = (_ffi.TcrtCamera * 1)(api.Camera().export())
    rgb = np.empty(4 * 4 * 3, F32)
    assert lib.tcrt_render_views(None, C.byref(p), 1, cams, rgb.ctypes.data, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_views_device(None, 0, C.byref(p), 1, cams, rgb.ctypes.data, None, None) == _ffi.TCRT_ERR_INVALID


def test_aim_reproduces_the_reference_cameras():
    assert np.array_equal(cam_bits(api.Camera().aim(*DEFAULT_POSE).export()), cam_bits(api.Camera().export()))
    tm = api.Camera()
    tm.setSceneTwoMirrors()
    assert np.array_equal(cam_bits(api.Camera().aim(*TWO_MIRRORS_POSE).export()), cam_bits(tm.export()))
    # aim keeps the screen size and is the same arithmetic wherever it is called
    c = api.Camera()
    c.setSceneTwoMirrors()
    assert np.array_equal(cam_bits(c.aim(*DEFAULT_POSE).export()), cam_bits(api.Camera().export()))


def test_aimed_cameras_render_through_the_oracle():
    scene, cam = make_scene("default")
    flat = scene.flatten()
    p = api.default_params(24, 16, 8)
    ref, cnt = O.render(flat, cam.export(), p)
    img, cnt2 = O.render(flat, api.Camera().aim(*DEFAULT_POSE).export(), p)
    assert_bit_identical(img, ref, "aimed default camera")
    assert cnt == cnt2
    frames, colours = [], []
    for c in orbit_cameras((-1.0, -1.0, 2.0), 3.0, 1.0, 4) + cube_cameras((-1.0, -1.0, 2.5)):
        img, cnt = O.render(flat, c, p)
        assert np.isfinite(img).all() and cnt["rays_primary"] == 24 * 16
        colours.append(len(np.unique(img.reshape(-1, 3), axis=0)))
        frames.append(img)
    assert min(colours[:4]) > 4 and sum(n > 4 for n in colours[4:]) >= 3, colours   # the views see the scene
    for a in range(len(frames)):
        for b in range(a):
            assert not np.array_equal(bits(frames[a]), bits(frames[b])), (a, b)


# ---- on the GPU --------------------------------------------------------------------------------------------------------------

def _view_size(depth):
    return (20, 16) if depth > 64 else (24, 16)


@gpu
@pytest.mark.parametrize("name", NAMES)
def test_views_of_every_dispatch_class(gpu_ctx, pair_ctx, name):
    s, flat, c = _upload(gpu_ctx, name)
    pair_ctx.upload_flat(flat, c)
    for depth in DEPTHS:
        p = api.default_params(*_view_size(depth), depth)
        check_views(gpu_ctx, flat, p, three_views(c), f"{name} d{depth}", pair=pair_ctx)


@gpu
@pytest.mark.parametrize("spec,w,h,d", [("default", 64, 48, 50), ("two_mirrors", 48, 40, 50), ("synth256", 64, 48, 10),
                                        ("lattice:1:4", 48, 32, 8)])
def test_views_of_named_scenes(gpu_ctx, pair_ctx, spec, w, h, d):
    scene, cam = make_scene(spec)
    flat, c = scene.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    pair_ctx.upload_flat(flat, c)
    if spec == "synth256":
        assert gpu_ctx.scene_structures()["grid_cells"] > 0
    check_views(gpu_ctx, flat, api.default_params(w, h, d), three_views(c) + [moved(c, (.1, .1, .1), fov=1.3)], spec,
                pair=pair_ctx)


@gpu
def test_orbit_and_cube_map_views(gpu_ctx, pair_ctx):
    for spec, centre in (("default", (-1.0, -1.0, 2.0)), ("synth256", (0.5, 0.5, 0.5))):
        scene, cam = make_scene(spec)
        flat = scene.flatten()
        gpu_ctx.upload_flat(flat, cam.export())
        pair_ctx.upload_flat(flat, cam.export())
        p = api.default_params(32, 24, 10)
        check_views(gpu_ctx, flat, p, orbit_cameras(centre, 3.0, 1.0, 5), f"{spec} orbit", pair=pair_ctx)
        check_views(gpu_ctx, flat, p, cube_cameras(centre), f"{spec} cube map", pair=pair_ctx)


@gpu
def test_degenerate_cameras(gpu_ctx, pair_ctx):
    """Cameras tcrt_set_camera accepts without a check: eye rays of 0/0 (NaN directions miss everything: the null colour),
    a NaN eye, an infinite screen, a screen of 1e30 (the direction's length overflows: zero directions)."""
    scene, cam = make_scene("default")
    flat, c = scene.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    pair_ctx.upload_flat(flat, c)
    flat_cam = copy_cam(c)                  # every eye ray is 0/0
    for k in range(3):
        flat_cam.horizontal[k] = flat_cam.vertical[k] = 0.0
        flat_cam.screen_origin[k] = flat_cam.eye[k]
    nan_cam = copy_cam(c)
    nan_cam.eye[0] = float("nan")
    inf_cam = copy_cam(c)
    inf_cam.screen_width = float("inf")
    huge_cam = copy_cam(c)
    huge_cam.screen_width = huge_cam.screen_height = 1e30
    p = api.default_params(16, 8, 8)
    got, _ = check_views(gpu_ctx, flat, p, [flat_cam, c, nan_cam, inf_cam, huge_cam], "degenerate",
                         pair=pair_ctx)
    assert (bits(got[0]) == bits(np.full(3, .75, F32))).all()


@gpu
@pytest.mark.parametrize("w,h,v", [(13, 11, 3), (1, 1, 1), (1, 9, 5), (7, 1, 3), (16, 8, 300)])
def test_view_shapes(gpu_ctx, pair_ctx, w, h, v):
    scene, cam = make_scene("two_mirrors")
    flat, c = scene.flatten(), cam.export()
    gpu_ctx.upload_flat(flat, c)
    pair_ctx.upload_flat(flat, c)
    cams = [moved(c, (.02 * (k % 17), -.01 * (k % 5), .005 * k)) for k in range(v)]
    got, st = check_views(gpu_ctx, flat, api.default_params(w, h, 20), cams, f"{v} x {w}x{h}", oracle=v <= 5,
                          pair=pair_ctx)
    assert st.gpu_launches == 1 and st.bands == [(0, v * w)]


@gpu
@pytest.mark.parametrize("w,h,v", [(3000, 1024, 3), (2048, 1024, 3), (1283, 2048, 4)])
def test_views_in_several_pieces(gpu_ctx, w, h, v):
    """Pieces of 4 Mi pixels: with H = 1024, 4096 columns, so boundaries inside views (3000 x 3: at 4096 and 8192), on a
    view boundary (2048 x 3: at 4096), and, with W % 4 != 0, of 2048 columns inside views."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    p = api.default_params(w, h, 3)
    cams = three_views(c) + [moved(c, (.05, .05, 0.0))] * (v - 3)
    got, st = check_views(gpu_ctx, None, p, cams, f"{v} x {w}x{h}", oracle=False)
    per = PIECE // h
    per -= per % 4 if w % 4 == 0 else 0
    assert st.gpu_launches == (v * w + per - 1) // per >= 2


@gpu
def test_rgb8_views(gpu_ctx):
    scene, cam = make_scene("two_mirrors")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    cams = three_views(c)
    lib = _ffi.load()
    for w, h in ((40, 32), (13, 11)):
        p = api.default_params(w, h, 30)
        rgb, st = gpu_ctx.render_views(p, cams)
        rgb = rgb.copy()
        q, st8 = gpu_ctx.render_views_rgb8(p, cams)
        assert np.array_equal(q, quant8(rgb).astype(np.uint8))
        assert st8.gpu_launches == 2 and _counters(st8) == _counters(st)
        frames = []
        for cc in cams:
            gpu_ctx.set_camera(cc)
            f8, _ = gpu_ctx.render_rgb8(p)
            frames.append(f8.copy())
        assert np.array_equal(q, np.stack(frames))
        # both outputs in one call
        both_f = np.empty_like(rgb)
        both_q = np.empty_like(q)
        table = api._camera_table(cams)
        stc = _ffi.TcrtStats()
        assert lib.tcrt_render_views(gpu_ctx._h, C.byref(p), 3, table, both_f.ctypes.data, both_q.ctypes.data,
                                     C.byref(stc)) == _ffi.TCRT_OK
        assert np.array_equal(bits(both_f), bits(rgb)) and np.array_equal(both_q, q)
        assert stc.gpu_launches == 2


GUARD = 64


@gpu
def test_destinations(gpu_ctx):
    """Pinned and pageable destinations with guard words, and the device form with torch tensors: identical bits."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    cams = three_views(c) + [moved(c, (.2, .2, .2))]
    p = api.default_params(320, 240, 8)
    ref, st_ref = gpu_ctx.render_views(p, cams)
    ref = ref.copy()
    ref8, _ = gpu_ctx.render_views_rgb8(p, cams)
    ref8 = ref8.copy()
    shape = (4, 320, 240, 3)
    bufs = []

    def pinned(dtype):
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        hb = api.HostBuffer(nbytes + 2 * GUARD)
        bufs.append(hb)
        a = hb.array(np.uint8, (hb.nbytes,))
        a[:] = 0xA5
        return a[GUARD:GUARD + nbytes].view(dtype).reshape(shape), a

    def pageable(dtype):
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        a = np.full(nbytes + 2 * GUARD, 0xA5, np.uint8)
        return a[GUARD:GUARD + nbytes].view(dtype).reshape(shape), a

    for kind in (pinned, pageable):
        out, whole = kind(F32)
        got, st = gpu_ctx.render_views(p, cams, out=out)
        assert np.array_equal(bits(got), bits(ref)), kind.__name__
        assert (whole[:GUARD] == 0xA5).all() and (whole[-GUARD:] == 0xA5).all()
        assert _counters(st) == _counters(st_ref)
        out8, whole8 = kind(np.uint8)
        got8, _ = gpu_ctx.render_views_rgb8(p, cams, out=out8)
        assert np.array_equal(got8, ref8), kind.__name__
        assert (whole8[:GUARD] == 0xA5).all() and (whole8[-GUARD:] == 0xA5).all()
    import torch
    dev = torch.device("cuda:0")
    n = int(np.prod(shape))
    trgb = torch.full((n + 2 * GUARD,), 7.0, device=dev)
    t8 = torch.full((n + 2 * GUARD,), 7, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    for want_f, want_8 in ((True, False), (False, True), (True, True)):
        trgb.fill_(7.0)
        t8.fill_(7)
        torch.cuda.synchronize()
        st = gpu_ctx.render_views_device(p, cams, rgb=trgb[GUARD:].data_ptr() if want_f else 0,
                                         rgb8=t8[GUARD:].data_ptr() if want_8 else 0)
        assert _counters(st) == _counters(st_ref)
        assert st.gpu_launches == 1 + want_8
        f = trgb.cpu().numpy()
        q = t8.cpu().numpy()
        if want_f:
            assert np.array_equal(bits(f[GUARD:GUARD + n]), bits(ref).ravel())
        else:
            assert (f == 7.0).all()
        if want_8:
            assert np.array_equal(q[GUARD:GUARD + n], ref8.ravel())
        else:
            assert (q == 7).all()
        assert (f[:GUARD] == 7.0).all() and (f[GUARD + n:] == 7.0).all()
        assert (q[:GUARD] == 7).all() and (q[GUARD + n:] == 7).all()
    # a wrong slot, a host pointer, no output
    arr = np.empty(n, F32)
    for kw in (dict(rgb=trgb.data_ptr(), slot=1), dict(rgb=arr.ctypes.data), dict(rgb8=arr.ctypes.data), dict()):
        with pytest.raises(api.TcrtError) as e:
            gpu_ctx.render_views_device(p, cams, **kw)
        assert e.value.code == _ffi.TCRT_ERR_INVALID, kw


def expected_bands(n_cols, w, nd):
    unit = 4 if w % 4 == 0 else 1
    m = n_cols // unit
    cut = [(m // nd * i + m % nd * i // nd) * unit for i in range(nd + 1)]
    return [(cut[i], cut[i + 1]) for i in range(nd)]


@gpu
@pytest.mark.parametrize("n_bands", [2, 3])
def test_multi_device_views(gpu_ctx, n_bands):
    n_dev = api.device_count()
    scene, cam = make_scene("synth256")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    cams = three_views(c) + [moved(c, (.1, 0.0, .1))]
    multi = api.Context([i % n_dev for i in range(n_bands)])
    multi.upload(scene, cam)
    for w, h in ((64, 48), (37, 29)):
        p = api.default_params(w, h, 10)
        ref, st1 = gpu_ctx.render_views(p, cams)
        ref = ref.copy()
        got, st = multi.render_views(p, cams)
        assert np.array_equal(bits(got), bits(ref)), f"{n_bands} devices {w}x{h}"
        assert st.bands == expected_bands(4 * w, w, n_bands)
        assert _counters(st) == _counters(st1)
        q, _ = multi.render_views_rgb8(p, cams)
        assert np.array_equal(q, quant8(ref).astype(np.uint8))
    multi.close()


@gpu
def test_views_leave_the_frames_the_camera_and_the_cut_alone(gpu_ctx, tmp_path):
    scene, cam = make_scene("two_mirrors")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    p = api.default_params(64, 48, 20)
    cams = three_views(moved(c, (.4, -.3, .2)))
    cut = gpu_ctx.balance_columns(p, 3)
    frame, _ = gpu_ctx.render(p)
    frame = frame.copy()
    gpu_ctx.write_ppm(p, str(tmp_path / "a.ppm"))
    ref, _ = gpu_ctx.render_views(p, cams)
    ref = ref.copy()
    buf = [api.HostBuffer(64 * 48 * 12) for _ in range(2)]
    outs = [b.array(F32, (64, 48, 3)) for b in buf]
    t = [gpu_ctx.render_async(p, 0, 64, outs[k]) for k in range(2)]
    got, _ = gpu_ctx.render_views(p, cams)                  # two frames in flight
    assert np.array_equal(bits(got), bits(ref)), "with two frames in flight"
    for k in range(2):
        gpu_ctx.wait(t[k])
        assert_bit_identical(outs[k], frame, "frame in flight")
    assert_bit_identical(gpu_ctx.download(np.empty_like(frame)), frame, "last render")
    gpu_ctx.write_ppm(p, str(tmp_path / "b.ppm"))
    assert (tmp_path / "a.ppm").read_bytes() == (tmp_path / "b.ppm").read_bytes()
    again, _ = gpu_ctx.render(p)                            # the ctx camera is still c
    assert_bit_identical(again, frame, "ctx camera")
    assert gpu_ctx.balance_columns(p, 3) == cut


@gpu
def test_error_codes(gpu_ctx):
    lib = _ffi.load()
    c = api.Camera().export()
    table = (_ffi.TcrtCamera * 2)(c, c)
    rgb = np.empty(2 * 4 * 4 * 3, F32)
    r = rgb.ctypes.data
    fresh = api.Context([0])
    with pytest.raises(api.TcrtError) as e:
        fresh.render_views(api.default_params(4, 4, 2), [c])
    assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
    fresh.close()
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    h = gpu_ctx._h
    p = api.default_params(4, 4, 2)
    assert lib.tcrt_render_views(h, None, 2, table, r, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_views(h, C.byref(p), 2, None, r, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_views(h, C.byref(p), 2, table, None, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_views(h, C.byref(p), -1, table, r, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_views_device(h, -1, C.byref(p), 2, table, r, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_views_device(h, 5, C.byref(p), 2, table, r, None, None) == _ffi.TCRT_ERR_INVALID
    for field, value in (("width", 0), ("height", -3), ("max_depth", -1)):
        bad = api.default_params(4, 4, 2)
        setattr(bad, field, value)
        assert lib.tcrt_render_views(h, C.byref(bad), 2, table, r, None, None) == _ffi.TCRT_ERR_INVALID, field
    deep = api.default_params(4, 4, 255)
    assert lib.tcrt_render_views(h, C.byref(deep), 2, table, r, None, None) == _ffi.TCRT_ERR_UNSUPPORTED
    wide = api.default_params(1 << 20, 1, 2)
    assert lib.tcrt_render_views(h, C.byref(wide), 1 << 11, table, r, None, None) == _ffi.TCRT_ERR_UNSUPPORTED
    st = _ffi.TcrtStats()
    assert lib.tcrt_render_views(h, C.byref(p), 0, None, r, None, C.byref(st)) == _ffi.TCRT_OK
    assert st.gpu_launches == 0 and st.rays_primary[0] == 0
    got, st = gpu_ctx.render_views(p, [])
    assert got.shape == (0, 4, 4, 3) and st.gpu_launches == 0


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
    std::vector<Camera> views(3);
    views[1].aim(vector3d(-4.f, -4.f, 1.5f), vector3d(.1f, -.08f, 0.f), vector3d(.08f, .1f, .01f));
    views[2].aim(vector3d(-3.f, -5.f, 2.f), vector3d(.1f, -.05f, 0.f), vector3d(.05f, .1f, -.02f));
    const int W = 48, H = 40;
    GpuRayTracer rt;
    RenderSettings rs;
    rs.width = W; rs.height = H; rs.max_depth = 50;
    std::vector<float> rgb(3 * W * H * 3);
    std::vector<unsigned char> rgb8(3 * W * H * 3);
    if (!rt.ok() || rt.setScene(scene, camera) || rt.renderViews(rs, views, rgb.data(), rgb8.data())) {
        fprintf(stderr, "%s\n", rt.lastError());
        return 1;
    }
    RenderSettings ss = rs;
    ss.samples = 2;
    printf("%d\n", rt.renderViews(ss, views, rgb.data()));
    tcrt_camera c2;
    views[2].exportTo(&c2);
    FILE* f = fopen("views.bin", "wb");
    if (!f) return 1;
    fwrite(rgb.data(), 4, rgb.size(), f);
    fwrite(rgb8.data(), 1, rgb8.size(), f);
    fwrite(&c2, sizeof c2, 1, f);
    return fclose(f) ? 1 : 0;
}
"""


@gpu
def test_cpp_render_views(gpu_ctx, tmp_path):
    src = tmp_path / "views.cpp"
    src.write_text(CPP_PROGRAM)
    libdir = os.path.join(ROOT, "tilecoderaytracer_b200")
    exe = tmp_path / "views"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), str(src),
                    "-L", libdir, "-ltcrt", f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert int(r.stdout.split()[-1]) == _ffi.TCRT_ERR_UNSUPPORTED      # samples != 1
    n = 3 * 48 * 40 * 3
    raw = (tmp_path / "views.bin").read_bytes()
    rgb = np.frombuffer(raw[:4 * n], F32).reshape(3, 48, 40, 3)
    rgb8 = np.frombuffer(raw[4 * n:5 * n], np.uint8).reshape(3, 48, 40, 3)
    c2 = _ffi.TcrtCamera.from_buffer_copy(raw[5 * n:])
    assert np.array_equal(cam_bits(c2), cam_bits(api.Camera().aim((-3.0, -5.0, 2.0), (.1, -.05, 0.0),
                                                                  (.05, .1, -.02)).export()))
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    c = cam.export()
    want, _ = per_view(gpu_ctx, api.default_params(48, 40, 50), [c, c, c2])
    assert np.array_equal(bits(rgb), bits(want))
    assert np.array_equal(rgb8, quant8(want).astype(np.uint8))
