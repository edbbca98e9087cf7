"""8-bit RGB frames (tcrt_render_rgb8, tcrt_render_columns_rgb8, tcrt_render_async_rgb8): each column chunk is quantised
on the GPU, q(c) = floor(clamp(c,0,1)*255 + 0.5), and 3 bytes per pixel cross the bus.  The byte frame must be exactly
quant8 of the float frame, which is itself bit-identical to the reference's; the float frame stays the last render."""
import ctypes as C
import copy
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import bits, make_scene, pixel_md5, quant8

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu


def q8(img):
    return quant8(img).astype(np.uint8)


def assert_bytes_equal(got, want, what=""):
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    bad = int((got != want).any(-1).sum())
    assert bad == 0, f"{what}: {bad} of {got.shape[0] * got.shape[1]} pixels differ"


# ---- no device needed ------------------------------------------------------------------------------------------------

def test_rgb8_entry_points_refuse_a_null_context():
    lib = _ffi.load()
    p = api.default_params(8, 8, 2)
    buf = np.zeros(8 * 8 * 3, np.uint8)
    dst = buf.ctypes.data_as(C.c_void_p)
    st = _ffi.TcrtStats()
    t = C.c_int(-1)
    assert lib.tcrt_render_rgb8(None, C.byref(p), dst, C.byref(st)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_columns_rgb8(None, C.byref(p), 0, 8, dst, C.byref(st)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_async_rgb8(None, C.byref(p), 0, 8, dst, C.byref(t)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_rgb8(None, None, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_async_rgb8(None, C.byref(p), 0, 8, None, None) == _ffi.TCRT_ERR_INVALID
    assert (buf == 0).all()


# ---- equal to the quantised reference ---------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("scene,w,h,d", [
    ("default", 500, 504, 50), ("default", 97, 61, 4), ("default", 1, 1, 50), ("two_mirrors", 96, 80, 50),
    ("synth256", 160, 128, 10), ("lattice:1:4", 160, 128, 12),
])
def test_rgb8_equals_quantised_float_frame_and_oracle(gpu_ctx, scene, w, h, d):
    s, cam = make_scene(scene)
    p = api.default_params(w, h, d)
    gpu_ctx.upload(s, cam)
    img, st = gpu_ctx.render(p)
    got, st8 = gpu_ctx.render_rgb8(p)
    assert got.dtype == np.uint8 and got.shape == (w, h, 3)
    assert_bytes_equal(got, q8(img), f"{scene} {w}x{h} d{d} vs quant8(float frame)")
    want, cnt = O.render(s.flatten(), cam.export(), p)
    assert_bytes_equal(got, q8(want), f"{scene} {w}x{h} d{d} vs quant8(oracle)")
    assert (st8.rays_primary, st8.rays_shadow, st8.rays_reflect) == (st.rays_primary, st.rays_shadow, st.rays_reflect)
    assert (st8.rays_primary, st8.rays_shadow, st8.rays_reflect) == (cnt["rays_primary"], cnt["rays_shadow"], cnt["rays_reflect"])
    assert st8.gpu_launches == st.gpu_launches + 1          # one chunk at these sizes: its render launch + one quantisation


@gpu
def test_rgb8_equals_quantised_golden_frames(gpu_ctx, golden, golden_frames):
    """The goldens were rendered by the reference program itself."""
    for key, m in golden["frames"].items():
        scene, cam = make_scene(m["scene"])
        gpu_ctx.upload(scene, cam)
        got, _ = gpu_ctx.render_rgb8(api.default_params(m["W"], m["H"], m["depth"]))
        assert_bytes_equal(got, q8(golden_frames[key]), key)


# ---- chunked and staged copies --------------------------------------------------------------------------------------

GUARD = 4096


def _check_band(render, want, what):
    """render(buf) writes the band into buf[:want.size]; twice, from two different fills, so that a byte which was not
    written cannot pass; the guard bytes behind the band must keep their fill."""
    for fill in (0xAB, 0x54):
        buf = render(fill)
        band = buf[:want.size].reshape(want.shape)
        assert_bytes_equal(band, want, f"{what}, fill {fill:#x}")
        assert (buf[want.size:] == fill).all(), f"{what}: a guard byte after the band was overwritten"


@gpu
@pytest.mark.parametrize("name,w,h,d", [("default", 1920, 1080, 5), ("default", 3840, 2160, 50), ("synth256", 1920, 1080, 10),
                                        ("default", 1920, 1081, 5)])
def test_rgb8_chunked_pinned_and_pageable_destinations(gpu_ctx, name, w, h, d):
    """Whole frames and column ranges.  [13, 1002) is 989 columns wide, not a multiple of the 4-column tile, so its chunks
    start at any column; with 1081 rows (3*1081 channels per column, not a multiple of 4) the chunks after the first start
    off the 16-byte alignment of the float frame and the quantiser runs its scalar head."""
    scene, cam = make_scene(name)
    p = api.default_params(w, h, d)
    gpu_ctx.upload(scene, cam)
    img, st = gpu_ctx.render(p)
    want = q8(img)
    del img
    for x0, x1 in ((0, w), (13, 1001), (13, 1002)):
        n = (x1 - x0) * h * 3
        hb = api.HostBuffer(n + GUARD)
        pinned = hb.array(np.uint8, (n + GUARD,))
        pageable = np.empty(n + GUARD, np.uint8)
        for kind, buf in (("pinned", pinned), ("pageable", pageable)):
            def render(fill, buf=buf):
                buf[:] = fill
                _, st8 = gpu_ctx.render_rgb8(p, x0, x1, out=buf[:n].reshape(x1 - x0, h, 3))
                assert st8.gpu_launches > 2, "expected a chunked render"
                if (x0, x1) == (0, w):
                    assert st8.rays == st.rays
                return buf
            _check_band(render, want[x0:x1], f"{name} {w}x{h} d{d} [{x0},{x1}) {kind}")
        del hb, pinned


@gpu
def test_staged_copy_of_a_single_chunk_band(gpu_ctx):
    """One column of 600 000 rows: enough pixels for the staged copy into pageable memory, one column, hence one chunk.
    The copy must wait for that chunk's render (and quantisation): every frame here differs from the one before it, so a
    copy that ran early would deliver the previous frame's bytes."""
    import copy as _copy

    scene, cam = make_scene("default")
    p = api.default_params(4, 600_000, 50)
    gpu_ctx.upload(scene, cam)
    hb = api.HostBuffer(600_000 * 12)
    for i in range(3):
        c = _copy.copy(cam.export())
        c.eye[0] += 0.1 * i
        gpu_ctx.set_camera(c)
        want, st_w = gpu_ctx.render(p, 1, 2, out=hb.array(np.float32, (1, 600_000, 3)))    # pinned: direct copies
        want = want.copy()
        got8 = np.full((1, 600_000, 3), 0xAB, np.uint8)
        _, st8 = gpu_ctx.render_rgb8(p, 1, 2, out=got8)
        assert st8.gpu_launches == st_w.gpu_launches + 1 and st8.rays == st_w.rays
        assert_bytes_equal(got8, q8(want), f"RGB8 frame {i}, one-chunk band, pageable")
        gotf = np.full((1, 600_000, 3), -1.0, np.float32)
        gpu_ctx.render(p, 1, 2, out=gotf)
        assert np.array_equal(bits(gotf), bits(want)), f"float frame {i}, one-chunk band, pageable"
    gpu_ctx.set_camera(cam.export())


@gpu
@pytest.mark.parametrize("n_bands", [4, 8])
def test_staged_copy_of_single_chunk_device_bands(gpu_ctx, n_bands):
    """A multi-device frame large enough to go through the pinned staging into pageable memory, whose device bands are each
    below 512 K pixels: such a band is rendered as ONE chunk, and its staged copy must still wait for that chunk's
    launches (1920x1080 on 4 or 8 devices: bands of about 480 or 240 columns).  With fewer GPUs visible the device ids
    repeat: several band states of the context share a GPU, each with its own streams and buffers."""
    n = api.device_count()
    devs = [i % n for i in range(n_bands)]
    scene, cam = make_scene("default")
    w, h = 1920, 1080
    p = api.default_params(w, h, 5)
    gpu_ctx.upload(scene, cam)
    want, st1 = gpu_ctx.render(p)
    multi = api.Context(devs)
    multi.upload(scene, cam)
    for i in range(3):                                    # fresh buffers first, then the rebalanced cuts
        got8 = np.full((w, h, 3), 0xAB, np.uint8)
        _, st = multi.render_rgb8(p, out=got8)
        assert st.n_devices == n_bands and st.rays == st1.rays
        assert min(b1 - b0 for b0, b1 in st.bands) * h < 2 * 256 * 1024, st.bands     # some band is one chunk
        assert_bytes_equal(got8, q8(want), f"RGB8 frame {i} on {n_bands} bands, pageable")
        gotf = np.full((w, h, 3), -1.0, np.float32)
        _, st = multi.render(p, out=gotf)
        assert st.rays == st1.rays
        assert np.array_equal(bits(gotf), bits(want)), f"float frame {i} on {n_bands} bands, pageable"
    multi.close()


@gpu
def test_rgb8_at_full_baseline_size(gpu_ctx):
    """synth256 7680x4320 depth 10 (the largest BASELINE frame)."""
    scene, cam = make_scene("synth256")
    p = api.default_params(7680, 4320, 10)
    gpu_ctx.upload(scene, cam)
    img, st = gpu_ctx.render(p)
    got, st8 = gpu_ctx.render_rgb8(p)
    assert st8.rays == st.rays
    for c0 in range(0, 7680, 960):
        assert_bytes_equal(got[c0:c0 + 960], q8(img[c0:c0 + 960]), f"synth256 8K columns [{c0},{c0 + 960})")


# ---- asynchronous frames --------------------------------------------------------------------------------------------

@gpu
def test_rgb8_and_float_async_frames_alternate(gpu_ctx, golden, tmp_path):
    scene, cam = make_scene("default")
    w, h = 320, 200
    p = api.default_params(w, h, 12)
    gpu_ctx.upload(scene, cam)
    cams = []
    for i in range(5):
        c = copy.copy(cam.export())
        c.eye[0] += 0.05 * i
        cams.append(c)
    want = []
    for c in cams:
        gpu_ctx.set_camera(c)
        img, st = gpu_ctx.render(p)
        want.append((img.copy(), st.rays))
    # frames 0, 2, 4 are RGB8, 1 and 3 float; a pinned buffer per frame
    hbs = [api.HostBuffer(w * h * (3 if i % 2 == 0 else 12)) for i in range(5)]
    outs = [hb.array(np.uint8 if i % 2 == 0 else np.float32, (w, h, 3)) for i, hb in enumerate(hbs)]

    def check(i, st):
        if i % 2 == 0:
            assert_bytes_equal(outs[i], q8(want[i][0]), f"async RGB8 frame {i}")
        else:
            assert np.array_equal(bits(outs[i]), bits(want[i][0])), f"async float frame {i}"
        assert st.rays == want[i][1]

    tickets = []
    for i, c in enumerate(cams):
        if len(tickets) == 2:
            j, t = tickets.pop(0)
            check(j, gpu_ctx.wait(t))
        gpu_ctx.set_camera(c)
        if i % 2 == 0:
            tickets.append((i, gpu_ctx.render_async_rgb8(p, 0, w, outs[i])))
        else:
            tickets.append((i, gpu_ctx.render_async(p, out=outs[i])))
        if len(tickets) == 2:
            with pytest.raises(api.TcrtError) as e:      # a third frame in flight is refused, in either format
                gpu_ctx.render_async_rgb8(p, 0, w, outs[0])
            assert e.value.code == _ffi.TCRT_ERR_INVALID
    for j, t in tickets:
        check(j, gpu_ctx.wait(t))
    # the last frame waited for was an RGB8 frame: download() gives its float frame
    got = np.empty((w, h, 3), np.float32)
    gpu_ctx.download(got)
    assert np.array_equal(bits(got), bits(want[4][0]))
    gpu_ctx.set_camera(cam.export())
    # and the writers see the float frame of an RGB8 frame: the reference's own file
    g = golden["md5"]["default_500x504_d50"]
    p = api.default_params(g["W"], g["H"], g["depth"])
    hb = api.HostBuffer(g["W"] * g["H"] * 3)
    out = hb.array(np.uint8, (g["W"], g["H"], 3))
    gpu_ctx.wait(gpu_ctx.render_async_rgb8(p, 0, g["W"], out))
    path = str(tmp_path / "raytracer_screen.txt")
    gpu_ctx.write_txt(p, path)
    txt = open(path, "rb").read()
    assert pixel_md5(txt) == g["pixel_md5"]
    frame = gpu_ctx.download(np.empty((g["W"], g["H"], 3), np.float32))
    assert_bytes_equal(out, q8(frame), "RGB8 of the reference's configuration")


# ---- clamping -------------------------------------------------------------------------------------------------------

@gpu
def test_rgb8_clamps_above_one_and_below_zero(gpu_ctx):
    # a light of intensity 12 seen directly: channels >= 10
    cam = api.Camera()
    s = api.Scene()
    s.addSphere((-2, -2, 2.0), .8).setAsLightSource(12.0)
    s.addInfinitePlane((0, 0, 0), (0, 0, 1), (1, 0, 0)).setCheckerBoard((1, 1, 1), (0, 0, 0), 3, 3)
    s.addSphere((0, 0, 1), 1.0).setColor(1, 0, 0).setReflectiveFactor(.7)
    p = api.default_params(160, 120, 6)
    gpu_ctx.upload(s, cam)
    img, _ = gpu_ctx.render(p)
    got, _ = gpu_ctx.render_rgb8(p)
    assert img.max() >= 10.0
    assert (got[img >= 1.0] == 255).all()
    assert_bytes_equal(got, q8(img), "intensity-12 light")
    # a lit sphere with a negative colour channel: negative floats
    s = api.Scene()
    s.addSphere((-2, -6, 12), .15).setAsLightSource(1.0)
    s.addInfinitePlane((0, 0, 0), (0, 0, 1), (1, 0, 0)).setCheckerBoard((1, 1, 1), (0, 0, 0), 3, 3)
    s.addSphere((0, 0, 1), 1.0).setColor(-1, .5, .5)
    gpu_ctx.upload(s, cam)
    img, _ = gpu_ctx.render(p)
    got, _ = gpu_ctx.render_rgb8(p)
    assert (img < 0).any()
    assert (got[img < 0] == 0).all()
    assert_bytes_equal(got, q8(img), "negative colour")


# ---- several GPUs in one context ------------------------------------------------------------------------------------

@gpu
def test_rgb8_multi_device_context_if_available(gpu_ctx):
    n = api.device_count()
    if n < 2:
        pytest.skip("one GPU visible")
    multi = api.Context(list(range(n)))
    for name, w, h, d in (("default", 640, 360, 8), ("default", 1920, 1080, 5)):
        scene, cam = make_scene(name)
        p = api.default_params(w, h, d)
        gpu_ctx.upload(scene, cam)
        one, st1 = gpu_ctx.render_rgb8(p)
        multi.upload(scene, cam)
        for _ in range(2):                                # the second frame is cut by the measured band times
            got, st = multi.render_rgb8(p)
            assert st.n_devices == n and st.rays == st1.rays
            assert_bytes_equal(got, one, f"{name} {w}x{h} d{d} on {n} GPUs")
        hb = api.HostBuffer(w * h * 3)
        pinned = hb.array(np.uint8, (w, h, 3))
        multi.render_rgb8(p, out=pinned)
        assert_bytes_equal(pinned, one, f"{name} {w}x{h} d{d} on {n} GPUs, pinned")
    multi.close()


# ---- errors ---------------------------------------------------------------------------------------------------------

@gpu
def test_rgb8_error_codes(gpu_ctx):
    lib = _ffi.load()
    fresh = api.Context([0])
    p = api.default_params(8, 8, 2)
    with pytest.raises(api.TcrtError) as e:
        fresh.render_rgb8(p)
    assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
    scene, cam = make_scene("default")
    fresh.upload(scene, cam)
    st = _ffi.TcrtStats()
    t = C.c_int(-1)
    assert lib.tcrt_render_rgb8(fresh._h, C.byref(p), None, C.byref(st)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_columns_rgb8(fresh._h, C.byref(p), 0, 8, None, C.byref(st)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_async_rgb8(fresh._h, C.byref(p), 0, 8, None, C.byref(t)) == _ffi.TCRT_ERR_INVALID
    for ticket in (0, 1):                                  # nothing was queued by the refused calls
        with pytest.raises(api.TcrtError) as e:
            fresh.wait(ticket)
        assert e.value.code == _ffi.TCRT_ERR_INVALID
    for x0, x1 in ((3, 3), (5, 2), (-1, 4), (0, 9)):
        buf = np.zeros(max(1, (x1 - x0)) * 8 * 3, np.uint8)
        rc = lib.tcrt_render_columns_rgb8(fresh._h, C.byref(p), x0, x1, buf.ctypes.data_as(C.c_void_p), C.byref(st))
        assert rc == _ffi.TCRT_ERR_INVALID, (x0, x1)
        rc = lib.tcrt_render_async_rgb8(fresh._h, C.byref(p), x0, x1, buf.ctypes.data_as(C.c_void_p), C.byref(t))
        assert rc == _ffi.TCRT_ERR_INVALID, (x0, x1)
        assert (buf == 0).all()
    got, _ = fresh.render_rgb8(p, 2, 6)                   # and the context still works
    assert got.shape == (4, 8, 3)
    fresh.close()


# ---- C++ -----------------------------------------------------------------------------------------------------------

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
    std::vector<unsigned char> px((size_t)rs.width * rs.height * 3);
    if (!rt.ok() || rt.setScene(scene, camera) || rt.renderRGB8(rs, px.data())) {
        fprintf(stderr, "%s\n", rt.lastError());
        return 1;
    }
    FILE* f = fopen("frame.rgb8", "wb");
    if (!f || fwrite(px.data(), 1, px.size(), f) != px.size()) return 1;
    return fclose(f) ? 1 : 0;
}
"""


@gpu
def test_cpp_render_rgb8(gpu_ctx, tmp_path):
    src = tmp_path / "render_rgb8.cpp"
    src.write_text(CPP_PROGRAM)
    libdir = os.path.join(ROOT, "tilecoderaytracer_b200")
    exe = tmp_path / "render_rgb8"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), str(src),
                    "-L", libdir, "-ltcrt", f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.fromfile(tmp_path / "frame.rgb8", dtype=np.uint8).reshape(200, 152, 3)
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    want, _ = gpu_ctx.render_rgb8(api.default_params(200, 152, 50))
    assert_bytes_equal(got, want, "GpuRayTracer::renderRGB8 vs Context.render_rgb8")
