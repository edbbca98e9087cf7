"""Primary-hit buffers (tcrt_hit_buffers, tcrt_device_hit_buffers) and picking (tcrt_pick): per pixel the object index,
distance and normal of the primary ray's nearest hit, computed on the GPU.  Every value is one the reference computes at
level 0 of calculatePixel, so the buffers are compared bit for bit with the pinned oracle's own nearest_hit and build_hit
(tests/oracle_hits.c), and the oracle extension itself is checked against frames rendered by the reference."""
import copy
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import bits, make_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
NAMES = ("object", "distance", "normal")


# ---- the oracle extension ---------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def hits_lib(tmp_path_factory):
    so = tmp_path_factory.mktemp("oracle_hits") / "liboracle_hits.so"
    subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", os.path.join(ROOT, "tests", "oracle_hits.c"),
                    "-o", str(so), "-lm"], check=True)
    lib = C.CDLL(str(so))
    lib.tcrt_oracle_primary_hits.restype = C.c_int
    lib.tcrt_oracle_primary_hits.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                             C.c_void_p, C.c_void_p, C.c_void_p]
    return lib


def primary_hits(lib, flat, cam, params, x0=0, x1=None, stride=1):
    """The oracle's primary hits of columns x0, x0+stride, ... < x1: {"object", "distance", "normal"}, x-major."""
    x1 = params.width if x1 is None else x1
    ncols = (x1 - x0 + stride - 1) // stride
    out = {"object": np.empty((ncols, params.height), np.int32), "distance": np.empty((ncols, params.height), np.float32),
           "normal": np.empty((ncols, params.height, 3), np.float32)}
    rc = lib.tcrt_oracle_primary_hits(C.byref(flat), C.byref(cam), C.byref(params), x0, x1, stride,
                                      *(out[k].ctypes.data_as(C.c_void_p) for k in NAMES))
    assert rc == 0
    return out


def _words(a):
    return np.ascontiguousarray(a).view(np.uint32)


def assert_hits_equal(got, want, what=""):
    for k in NAMES:
        assert got[k].shape == want[k].shape, f"{what} {k}: shape {got[k].shape} vs {want[k].shape}"
        diff = _words(got[k]) != _words(want[k])
        if k == "normal":
            diff = diff.any(-1)
        bad = int(diff.sum())
        assert bad == 0, f"{what} {k}: {bad} of {diff.size} pixels differ bitwise"


def scene_tables(flat):
    n = flat.n_objects
    info = np.ctypeslib.as_array(flat.obj_info, (n * 4,)).reshape(n, 4)
    surf = np.ctypeslib.as_array(flat.obj_surface, (n * 4,)).reshape(n, 4)
    mat = np.ctypeslib.as_array(flat.obj_material, (n * 4,)).reshape(n, 4)
    return info, surf, mat


def check_against_frame(flat, p, hits, frame, what):
    """A miss is the null colour and far_dist; an untextured light is its colour times its intensity
    (RayTracer.cpp:520-527).  Returns (misses, light pixels) checked."""
    obj = hits["object"]
    miss = obj == -1
    null = np.array(p.null_color[:], np.float32)
    assert (bits(frame[miss]) == bits(null)).all(), f"{what}: a miss is not the null colour"
    assert (_words(hits["distance"][miss]) == _words(np.float32(p.far_dist))).all(), f"{what}: a miss is not at far_dist"
    assert (_words(hits["normal"][miss]) == 0).all(), f"{what}: a miss has a normal"
    info, surf, mat = scene_tables(flat)
    light_rgb = surf[:, :3] * mat[:, 2:3]                      # float32 products
    untextured_light = (info[:, 2] != 0) & (info[:, 3] < 0)
    sel = ~miss & untextured_light[np.maximum(obj, 0)]
    assert (bits(frame[sel]) == bits(light_rgb[obj[sel]])).all(), f"{what}: a light pixel is not the light's colour"
    return int(miss.sum()), int(sel.sum())


# ---- no device needed ------------------------------------------------------------------------------------------------

def test_hit_entry_points_are_exported():
    lib = _ffi.load()
    for name in ("tcrt_hit_buffers", "tcrt_device_hit_buffers", "tcrt_pick"):
        assert hasattr(lib, name), name


def test_hit_entry_points_refuse_a_null_context():
    lib = _ffi.load()
    p = api.default_params(8, 8, 2)
    obj = np.full(64, 7, np.int32)
    dist = np.full(64, 7.0, np.float32)
    normal = np.full(64 * 3, 7.0, np.float32)
    st = _ffi.TcrtStats()
    ptrs = [a.ctypes.data_as(C.c_void_p) for a in (obj, dist, normal)]
    assert lib.tcrt_hit_buffers(None, C.byref(p), 0, 8, *ptrs, C.byref(st)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_hit_buffers(None, None, 0, 8, None, None, None, None) == _ffi.TCRT_ERR_INVALID
    xz = np.zeros(2, np.int32)
    assert lib.tcrt_pick(None, C.byref(p), 1, xz.ctypes.data_as(C.c_void_p), *ptrs) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_pick(None, C.byref(p), 0, None, None, None, None) == _ffi.TCRT_ERR_INVALID
    addr = [C.c_void_p(0x1234) for _ in range(3)]
    n = C.c_size_t(99)
    assert lib.tcrt_device_hit_buffers(None, 0, *(C.byref(a) for a in addr), C.byref(n)) == _ffi.TCRT_ERR_INVALID
    assert [a.value for a in addr] == [0x1234] * 3 and n.value == 99
    assert (obj == 7).all() and (dist == 7.0).all() and (normal == 7.0).all()


def test_oracle_hits_agree_with_the_reference_golden_frames(hits_lib, golden, golden_frames):
    """The goldens were rendered by the reference program itself (default, synth256, synth1024, two_mirrors, random and
    boxes scenes)."""
    misses = lights = 0
    for key, m in golden["frames"].items():
        scene, cam = make_scene(m["scene"])
        flat = scene.flatten()
        p = api.default_params(m["W"], m["H"], m["depth"])
        hits = primary_hits(hits_lib, flat, cam.export(), p)
        a, b = check_against_frame(flat, p, hits, golden_frames[key], key)
        misses += a
        lights += b
    assert misses > 0 and lights > 0, (misses, lights)


@pytest.mark.parametrize("spec,w,h,d", [("default", 120, 90, 5), ("two_mirrors", 64, 48, 20), ("lattice:1:4", 96, 72, 8),
                                        ("random:4:80", 96, 80, 6), ("boxes:3:14", 96, 80, 6)])
def test_oracle_hits_agree_with_oracle_renders(hits_lib, spec, w, h, d):
    scene, cam = make_scene(spec)
    flat = scene.flatten()
    p = api.default_params(w, h, d)
    hits = primary_hits(hits_lib, flat, cam.export(), p)
    frame, _ = O.render(flat, cam.export(), p)
    check_against_frame(flat, p, hits, frame, spec)
    # the parameters that only shading reads change nothing
    p2 = api.default_params(w, h, 0, shadows=False, reflections=False)
    p2.null_color[0] = 0.25
    assert_hits_equal(primary_hits(hits_lib, flat, cam.export(), p2), hits, f"{spec}: shading parameters")


def test_oracle_hits_light_scene(hits_lib):
    """Lights seen directly, one of them an intensity-12 light: the light pixels of the frame are colour x intensity."""
    cam = api.Camera()
    s = api.Scene()
    s.addSphere((-2, -2, 2.0), .8).setAsLightSource(12.0)
    s.addSphere((1, -3, 1.5), .5).setColor(.3, .6, .9).setAsLightSource(.7)
    s.addInfinitePlane((0, 0, 0), (0, 0, 1), (1, 0, 0)).setCheckerBoard((1, 1, 1), (0, 0, 0), 3, 3)
    s.addSphere((0, 0, 1), 1.0).setColor(1, 0, 0).setReflectiveFactor(.7)
    flat = s.flatten()
    p = api.default_params(160, 120, 6)
    hits = primary_hits(hits_lib, flat, cam.export(), p)
    frame, _ = O.render(flat, cam.export(), p)
    _, lights = check_against_frame(flat, p, hits, frame, "light scene")
    assert lights > 0


# ---- bit-exact against the oracle --------------------------------------------------------------------------------------

def gpu_and_oracle_hits(ctx, lib, flat, cam, p):
    ctx.upload_flat(flat, cam)
    got, st = ctx.hit_buffers(p)
    return got, st, primary_hits(lib, flat, cam, p)


@gpu
@pytest.mark.parametrize("spec,w,h,grid", [
    ("default", 500, 504, False), ("two_mirrors", 96, 80, False), ("synth256", 160, 128, True), ("synth1024", 160, 128, False),
    ("boxes:3:14", 128, 96, False), ("boxes:7:9", 128, 96, False), ("random:15:90", 136, 104, False),
    ("lattice:1:4", 160, 128, True),
])
def test_hit_buffers_equal_the_oracle(gpu_ctx, hits_lib, spec, w, h, grid):
    scene, cam = make_scene(spec)
    p = api.default_params(w, h, 7)
    got, st, want = gpu_and_oracle_hits(gpu_ctx, hits_lib, scene.flatten(), cam.export(), p)
    if grid:      # the scene has a sphere grid; the hit kernel walks the BVH built alongside it
        assert gpu_ctx.scene_structures()["grid_cells"] > 0
    assert_hits_equal(got, want, f"{spec} {w}x{h}")
    assert (got["object"] >= 0).any()
    if spec == "two_mirrors":
        assert scene.getObjectCount() == 3920


@gpu
@pytest.mark.parametrize("case", ["far_camera", "inside_sphere"])
def test_hit_buffers_sphere_grid_edge_cases(gpu_ctx, hits_lib, case):
    from test_gpu_parity import _lattice, _lights_and_ground

    cam = api.Camera()
    c = cam.export()
    s = api.Scene()
    _lights_and_ground(s)
    w, h = 128, 96
    if case == "far_camera":
        _lattice(s, 6, 6, 3, 1.8, .75)
        for k in range(3):
            shift = 600.0 * (.62, .78, .08)[k]
            c.eye[k] -= shift
            c.screen_origin[k] -= shift
        w, h = 96, 64
    else:
        _lattice(s, 5, 5, 3, 1.8, .75)
        eye = (-3 + 1.8 * 2 + .1, -1 + 1.8 * 2 - .2, .8 + 1.8)       # inside the sphere (2, 2, 1)
        for k in range(3):
            delta = eye[k] - c.eye[k]
            c.eye[k] += delta
            c.screen_origin[k] += delta
    p = api.default_params(w, h, 8)
    got, _, want = gpu_and_oracle_hits(gpu_ctx, hits_lib, s.flatten(), c, p)
    assert gpu_ctx.scene_structures()["grid_cells"] > 0
    assert_hits_equal(got, want, case)
    if case == "inside_sphere":
        assert (got["distance"] < 0).any(), "the sphere around the eye must win with a negative distance"


@gpu
def test_hit_buffers_4k_columns_at_a_stride(gpu_ctx, hits_lib):
    scene, cam = make_scene("default")
    p = api.default_params(3840, 2160, 50)
    gpu_ctx.upload(scene, cam)
    got, st = gpu_ctx.hit_buffers(p)
    want = primary_hits(hits_lib, scene.flatten(), cam.export(), p, 0, 3840, 97)
    assert_hits_equal({k: v[::97] for k, v in got.items()}, want, "default 4K, every 97th column")
    assert st.rays_primary == 3840 * 2160


# ---- bands, picking, destinations ---------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("w,h", [(256, 160), (203, 101)])
def test_hit_buffer_bands_concatenate_to_the_frame(gpu_ctx, hits_lib, w, h):
    """256x160 is tiled (4x8 tiles); 203x101 and the bands below are not, and take the column-by-column mapping."""
    scene, cam = make_scene("default")
    p = api.default_params(w, h, 5)
    gpu_ctx.upload(scene, cam)
    whole, _ = gpu_ctx.hit_buffers(p)
    assert_hits_equal(whole, primary_hits(hits_lib, scene.flatten(), cam.export(), p), f"{w}x{h}")
    cuts = (0, 70, 151, w)
    parts = [gpu_ctx.hit_buffers(p, a, b)[0] for a, b in zip(cuts[:-1], cuts[1:])]
    assert_hits_equal({k: np.concatenate([q[k] for q in parts]) for k in NAMES}, whole, f"{w}x{h}: three bands")
    one, st = gpu_ctx.hit_buffers(p, 77, 78)
    assert st.bands == [(77, 78)]
    assert_hits_equal(one, {k: v[77:78] for k, v in whole.items()}, f"{w}x{h}: one column")
    odd, _ = gpu_ctx.hit_buffers(p, 13, 26)      # 13 columns
    assert_hits_equal(odd, {k: v[13:26] for k, v in whole.items()}, f"{w}x{h}: 13 columns")


@gpu
def test_pick_equals_the_buffers(gpu_ctx):
    scene, cam = make_scene("two_mirrors")
    w, h = 320, 240
    p = api.default_params(w, h, 5)
    gpu_ctx.upload(scene, cam)
    whole, _ = gpu_ctx.hit_buffers(p)
    rng = np.random.default_rng(5)
    xs = np.concatenate([[0, w - 1, 0, w - 1], rng.integers(0, w, 1000)])
    zs = np.concatenate([[0, 0, h - 1, h - 1], rng.integers(0, h, 1000)])
    obj, dist, normal = gpu_ctx.pick(p, xs, zs)
    assert np.array_equal(obj, whole["object"][xs, zs])
    assert np.array_equal(_words(dist), _words(whole["distance"][xs, zs]))
    assert np.array_equal(_words(normal), _words(whole["normal"][xs, zs]))
    # every pixel once, in a shuffled order (more than one claim per warp, and a partial last claim)
    order = rng.permutation(w * h)
    obj, dist, normal = gpu_ctx.pick(p, order // h, order % h)
    assert np.array_equal(obj, whole["object"].reshape(-1)[order])
    assert np.array_equal(_words(normal), _words(whole["normal"].reshape(-1, 3)[order]))
    # n = 0, and single outputs
    lib = _ffi.load()
    assert lib.tcrt_pick(gpu_ctx._h, C.byref(p), 0, None, None, None, None) == 0
    xz = np.array([w - 1, h - 1], np.int32)
    d1 = np.full(1, -7.0, np.float32)
    assert lib.tcrt_pick(gpu_ctx._h, C.byref(p), 1, xz.ctypes.data_as(C.c_void_p), None, d1.ctypes.data_as(C.c_void_p), None) == 0
    assert _words(d1)[0] == _words(whole["distance"][w - 1, h - 1])
    # a pixel outside the frame: refused, nothing written
    for bad in ([w, 0], [0, h], [-1, 3], [3, -1]):
        xz = np.array([[1, 1], bad], np.int32)
        o = np.full(2, 0x5A5A5A5A, np.int32)
        d = np.full(2, -7.0, np.float32)
        n = np.full(6, -7.0, np.float32)
        rc = lib.tcrt_pick(gpu_ctx._h, C.byref(p), 2, xz.ctypes.data_as(C.c_void_p), o.ctypes.data_as(C.c_void_p),
                           d.ctypes.data_as(C.c_void_p), n.ctypes.data_as(C.c_void_p))
        assert rc == _ffi.TCRT_ERR_INVALID, bad
        assert (o == 0x5A5A5A5A).all() and (d == -7.0).all() and (n == -7.0).all()


GUARD = 4096


def _device_hits(ctx, slot=0):
    torch = pytest.importorskip("torch")
    o, d, n, cnt = ctx.device_hit_buffers(slot)

    def view(addr, typestr, count):
        class _Dev:
            __cuda_array_interface__ = {"shape": (count,), "typestr": typestr, "data": (addr, False), "version": 3}
        return torch.as_tensor(_Dev(), device="cuda").cpu().numpy()

    return {"object": view(o, "<i4", cnt), "distance": view(d, "<f4", cnt), "normal": view(n, "<f4", 3 * cnt)}, cnt


@gpu
def test_hit_buffer_destinations(gpu_ctx):
    """1920x1080 (above the 512 K-pixel staging threshold) into pinned and pageable memory, every non-empty subset of the
    three buffers: the requested ones arrive, the others and the guard bytes keep their 0xAB fill."""
    scene, cam = make_scene("default")
    w, h = 1920, 1080
    p = api.default_params(w, h, 5)
    gpu_ctx.upload(scene, cam)
    want, _ = gpu_ctx.hit_buffers(p)
    want = {k: v.copy() for k, v in want.items()}
    nbytes = {"object": w * h * 4, "distance": w * h * 4, "normal": w * h * 12}
    shapes = {"object": ((w, h), np.int32), "distance": ((w, h), np.float32), "normal": ((w, h, 3), np.float32)}
    pinned = {k: api.HostBuffer(nbytes[k] + GUARD) for k in NAMES}
    for kind in ("pinned", "pageable"):
        raw = {k: (pinned[k].array(np.uint8, (nbytes[k] + GUARD,)) if kind == "pinned" else np.empty(nbytes[k] + GUARD, np.uint8))
               for k in NAMES}
        for mask in range(1, 8):
            chosen = [k for i, k in enumerate(NAMES) if mask >> i & 1]
            for k in NAMES:
                raw[k][:] = 0xAB
            out = {k: raw[k][:nbytes[k]].view(shapes[k][1]).reshape(shapes[k][0]) for k in chosen}
            got, st = gpu_ctx.hit_buffers(p, out=out)
            assert sorted(got) == sorted(chosen)
            for k in NAMES:
                if k in chosen:
                    assert np.array_equal(_words(got[k]), _words(want[k])), f"{kind} {chosen}: {k}"
                    assert (raw[k][nbytes[k]:] == 0xAB).all(), f"{kind} {chosen}: guard bytes after {k}"
                else:
                    assert (raw[k] == 0xAB).all(), f"{kind} {chosen}: {k} was not requested but written"
            assert st.gpu_launches == 1 and st.rays_primary == w * h
    st = gpu_ctx.hit_buffers_device(p)
    assert st.d2h_ms == [0.0]
    dev, cnt = _device_hits(gpu_ctx)
    assert cnt == w * h
    for k in NAMES:
        assert np.array_equal(_words(dev[k]), _words(want[k].reshape(-1))), f"device-only {k}"


# ---- non-interference ---------------------------------------------------------------------------------------------------

@gpu
def test_hit_buffers_leave_the_last_render_alone(gpu_ctx, tmp_path):
    scene, cam = make_scene("default")
    w, h = 320, 200
    p = api.default_params(w, h, 12)
    gpu_ctx.upload(scene, cam)
    a, _ = gpu_ctx.render(p)
    a = a.copy()
    txt_a = gpu_ctx.format_txt()
    gpu_ctx.write_ppm(p, str(tmp_path / "a.ppm"))
    lib = _ffi.load()
    ptr_a, n_a = C.c_void_p(), C.c_size_t()
    assert lib.tcrt_device_frame(gpu_ctx._h, 0, C.byref(ptr_a), C.byref(n_a)) == 0
    gpu_ctx.hit_buffers(api.default_params(640, 360, 3))
    gpu_ctx.hit_buffers(p, 10, 20)
    gpu_ctx.pick(p, [1, 2], [3, 4])
    got = gpu_ctx.download(np.empty((w, h, 3), np.float32))
    assert np.array_equal(bits(got), bits(a))
    assert gpu_ctx.format_txt() == txt_a
    gpu_ctx.write_ppm(p, str(tmp_path / "b.ppm"))
    assert (tmp_path / "a.ppm").read_bytes() == (tmp_path / "b.ppm").read_bytes()
    ptr, n = C.c_void_p(), C.c_size_t()
    assert lib.tcrt_device_frame(gpu_ctx._h, 0, C.byref(ptr), C.byref(n)) == 0
    assert (ptr.value, n.value) == (ptr_a.value, n_a.value)


@gpu
def test_hit_buffers_with_two_frames_in_flight(gpu_ctx, hits_lib):
    scene, cam = make_scene("default")
    w, h = 640, 360
    p = api.default_params(w, h, 20)
    gpu_ctx.upload(scene, cam)
    cams = []
    for i in range(2):
        c = copy.copy(cam.export())
        c.eye[0] += 0.1 * i
        cams.append(c)
    want = []
    for c in cams:
        gpu_ctx.set_camera(c)
        want.append(gpu_ctx.render(p)[0].copy())
    hbs = [api.HostBuffer(w * h * 12) for _ in range(2)]
    outs = [hb.array(np.float32, (w, h, 3)) for hb in hbs]
    tickets = []
    for c, o in zip(cams, outs):
        o[:] = -1.0
        gpu_ctx.set_camera(c)
        tickets.append(gpu_ctx.render_async(p, out=o))
    hits, _ = gpu_ctx.hit_buffers(p)              # the camera of the last set_camera
    with pytest.raises(api.TcrtError):            # still two frames in flight
        gpu_ctx.render_async(p, out=outs[0])
    for t, o, wnt in zip(tickets, outs, want):
        gpu_ctx.wait(t)
        assert np.array_equal(bits(o), bits(wnt))
    got = gpu_ctx.download(np.empty((w, h, 3), np.float32))
    assert np.array_equal(bits(got), bits(want[1]))
    assert_hits_equal(hits, primary_hits(hits_lib, scene.flatten(), cams[1], p), "hit buffers between async frames")
    gpu_ctx.set_camera(cam.export())


@gpu
def test_hit_buffers_follow_set_camera(gpu_ctx, hits_lib):
    scene, cam = make_scene("synth256")
    p = api.default_params(192, 128, 4)
    gpu_ctx.upload(scene, cam)
    c = copy.copy(cam.export())
    for k in range(3):
        c.eye[k] += (.4, -.3, .2)[k]
        c.screen_origin[k] += (.4, -.3, .2)[k]
    gpu_ctx.set_camera(c)
    got, _ = gpu_ctx.hit_buffers(p)
    assert_hits_equal(got, primary_hits(hits_lib, scene.flatten(), c, p), "moved camera")
    obj, _, _ = gpu_ctx.pick(p, [100], [60])
    assert obj[0] == got["object"][100, 60]
    gpu_ctx.set_camera(cam.export())


# ---- stats and errors ----------------------------------------------------------------------------------------------------

@gpu
def test_hit_buffer_stats_and_errors(gpu_ctx):
    lib = _ffi.load()
    fresh = api.Context([0])
    p = api.default_params(64, 48, 2)
    for call in (lambda: fresh.hit_buffers(p), lambda: fresh.hit_buffers_device(p), lambda: fresh.pick(p, [1], [1])):
        with pytest.raises(api.TcrtError) as e:
            call()
        assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
    with pytest.raises(api.TcrtError) as e:
        fresh.device_hit_buffers(0)
    assert e.value.code == _ffi.TCRT_ERR_NO_FRAME
    scene, cam = make_scene("default")
    fresh.upload(scene, cam)
    st = _ffi.TcrtStats()
    for x0, x1 in ((3, 3), (5, 2), (-1, 4), (0, 65)):
        buf = np.zeros(64 * 48, np.int32)
        rc = lib.tcrt_hit_buffers(fresh._h, C.byref(p), x0, x1, buf.ctypes.data_as(C.c_void_p), None, None, C.byref(st))
        assert rc == _ffi.TCRT_ERR_INVALID, (x0, x1)
        assert (buf == 0).all()
    with pytest.raises(api.TcrtError) as e:
        fresh.device_hit_buffers(0)
    assert e.value.code == _ffi.TCRT_ERR_NO_FRAME
    _, st = fresh.hit_buffers(p, 8, 40)
    assert st.n_devices == 1 and st.bands == [(8, 40)]
    assert (st.rays_primary, st.rays_shadow, st.rays_reflect, st.gpu_launches) == (32 * 48, 0, 0, 1)
    assert st.render_ms[0] > 0 and st.d2h_ms[0] >= 0
    _, _, _, cnt = fresh.device_hit_buffers(0)
    assert cnt == 32 * 48
    with pytest.raises(api.TcrtError) as e:
        fresh.device_hit_buffers(1)
    assert e.value.code == _ffi.TCRT_ERR_INVALID
    fresh.close()


# ---- C++ ----------------------------------------------------------------------------------------------------------------

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
    GpuRayTracer rt;
    RenderSettings rs;
    rs.width = 200; rs.height = 152; rs.max_depth = 50;
    const size_t n = (size_t)rs.width * rs.height;
    std::vector<int> obj(n);
    std::vector<float> dist(n), normal(3 * n);
    if (!rt.ok() || rt.setScene(scene, camera) || rt.hitBuffers(rs, obj.data(), dist.data(), normal.data())) {
        fprintf(stderr, "%s\n", rt.lastError());
        return 1;
    }
    int po = -2;
    float pd = 0.f, pn[3] = {0.f, 0.f, 0.f};
    if (rt.pick(rs, 150, 40, &po, &pd, pn)) return 1;
    RenderSettings ss = rs;
    ss.samples = 2;
    if (rt.pick(ss, 150, 40, &po) != TCRT_ERR_UNSUPPORTED || rt.hitBuffers(ss, obj.data(), NULL, NULL) != TCRT_ERR_UNSUPPORTED)
        return 2;
    FILE* f = fopen("hits.bin", "wb");
    if (!f || fwrite(obj.data(), 4, n, f) != n || fwrite(dist.data(), 4, n, f) != n || fwrite(normal.data(), 4, 3 * n, f) != 3 * n ||
        fwrite(&po, 4, 1, f) != 1 || fwrite(&pd, 4, 1, f) != 1 || fwrite(pn, 4, 3, f) != 3)
        return 1;
    return fclose(f) ? 1 : 0;
}
"""


@gpu
def test_cpp_hit_buffers_and_pick(gpu_ctx, tmp_path):
    src = tmp_path / "hits.cpp"
    src.write_text(CPP_PROGRAM)
    libdir = os.path.join(ROOT, "tilecoderaytracer_b200")
    exe = tmp_path / "hits"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), str(src),
                    "-L", libdir, "-ltcrt", f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    w, h = 200, 152
    raw = np.fromfile(tmp_path / "hits.bin", dtype=np.uint32)
    n = w * h
    got = {"object": raw[:n].view(np.int32).reshape(w, h), "distance": raw[n:2 * n].view(np.float32).reshape(w, h),
           "normal": raw[2 * n:5 * n].view(np.float32).reshape(w, h, 3)}
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    want, _ = gpu_ctx.hit_buffers(api.default_params(w, h, 50))
    assert_hits_equal(got, want, "GpuRayTracer::hitBuffers vs Context.hit_buffers")
    tail = raw[5 * n:]
    assert tail[0].view(np.int32) == want["object"][150, 40]
    assert tail[1] == _words(want["distance"][150, 40])
    assert np.array_equal(tail[2:5], _words(want["normal"][150, 40]))


# ---- several GPUs in one context -------------------------------------------------------------------------------------------

@gpu
def test_hit_buffers_multi_device_context_if_available(gpu_ctx):
    n = api.device_count()
    if n < 2:
        pytest.skip("one GPU visible")
    multi = api.Context(list(range(n)))
    scene, cam = make_scene("default")
    for w, h in ((640, 360), (1920, 1080)):
        p = api.default_params(w, h, 5)
        gpu_ctx.upload(scene, cam)
        one, _ = gpu_ctx.hit_buffers(p)
        multi.upload(scene, cam)
        got, st = multi.hit_buffers(p)
        assert st.n_devices == n and st.rays_primary == w * h and st.gpu_launches == n
        assert_hits_equal(got, one, f"{w}x{h} on {n} GPUs")
        obj, _, _ = multi.pick(p, [w - 1], [h - 1])
        assert obj[0] == one["object"][w - 1, h - 1]
    multi.close()
