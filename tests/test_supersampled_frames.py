"""Supersampled frames (tcrt_render_columns_ss & co.): ss x ss samples per pixel, box-filtered on the GPU.  Sample (i, j) of
output pixel (x, z) is the reference's pixel (ss*x+i, ss*z+j) at (ss*W, ss*H), so a supersampled frame must be exactly
resolve() below of a frame that is itself bit-identical to the reference's: the goldens the reference program wrote,
the oracle, or the plain render at the sample size."""
import ctypes as C
import copy
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

from _util import assert_bit_identical, bits, make_scene, pixel_md5, quant8

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu

SS_ENTRY_POINTS = ("tcrt_render_columns_ss", "tcrt_render_columns_ss_rgb8", "tcrt_render_async_ss",
                   "tcrt_render_async_ss_rgb8")


def resolve(samples, ss):
    """The contract's box filter in float32: acc = sample(0,0), then acc += sample(i,j) for i (outer), j (inner), then one
    division by ss*ss.  samples: (ss*W, ss*H, 3) x-major."""
    s = np.asarray(samples, dtype=np.float32)
    assert s.shape[0] % ss == 0 and s.shape[1] % ss == 0, s.shape
    acc = s[0::ss, 0::ss].copy()
    for i in range(ss):
        for j in range(ss):
            if i or j:
                acc = acc + s[i::ss, j::ss]
    return acc / np.float32(ss * ss)


def q8(img):
    return quant8(img).astype(np.uint8)


def assert_bytes_equal(got, want, what=""):
    assert got.shape == want.shape, f"{what}: shape {got.shape} vs {want.shape}"
    bad = int((got != want).any(-1).sum())
    assert bad == 0, f"{what}: {bad} of {got.shape[0] * got.shape[1]} pixels differ"


def sample_params(p, ss):
    return api.default_params(ss * p.width, ss * p.height, p.max_depth)


# ---- no device needed ------------------------------------------------------------------------------------------------

def test_ss_symbols_are_exported():
    lib = C.CDLL(_ffi.LIB_PATH)
    for name in SS_ENTRY_POINTS:
        assert hasattr(lib, name), name


def test_ss_entry_points_refuse_a_null_context():
    lib = _ffi.load()
    p = api.default_params(8, 8, 2)
    f = np.zeros(8 * 8 * 3, np.float32)
    b = np.zeros(8 * 8 * 3, np.uint8)
    st = _ffi.TcrtStats()
    t = C.c_int(-1)
    for ss in (1, 2):
        assert lib.tcrt_render_columns_ss(None, C.byref(p), ss, 0, 8, f.ctypes.data_as(C.c_void_p), C.byref(st)) == \
            _ffi.TCRT_ERR_INVALID
        assert lib.tcrt_render_columns_ss_rgb8(None, C.byref(p), ss, 0, 8, b.ctypes.data_as(C.c_void_p), C.byref(st)) == \
            _ffi.TCRT_ERR_INVALID
        assert lib.tcrt_render_async_ss(None, C.byref(p), ss, 0, 8, f.ctypes.data_as(C.c_void_p), C.byref(t)) == \
            _ffi.TCRT_ERR_INVALID
        assert lib.tcrt_render_async_ss_rgb8(None, C.byref(p), ss, 0, 8, b.ctypes.data_as(C.c_void_p), C.byref(t)) == \
            _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_columns_ss(None, None, 2, 0, 8, None, None) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_async_ss_rgb8(None, C.byref(p), 2, 0, 8, None, None) == _ffi.TCRT_ERR_INVALID
    assert (f == 0).all() and (b == 0).all() and t.value == -1


def test_numpy_resolve_follows_the_contract_order():
    """resolve() is the sequential float32 sum, not a pairwise one: on these values the two orders differ."""
    s = np.zeros((2, 2, 3), np.float32)
    s[0, 0], s[0, 1], s[1, 0], s[1, 1] = 1.0, 2.0 ** -24, 2.0 ** -24, 2.0 ** -24
    seq = ((np.float32(1.0) + np.float32(2.0 ** -24)) + np.float32(2.0 ** -24)) + np.float32(2.0 ** -24)
    assert resolve(s, 2)[0, 0, 0] == seq / np.float32(4)
    assert seq != np.float32(1.0) + np.float32(3 * 2.0 ** -24)     # the values do tell the orders apart
    assert resolve(s, 1) is not s and np.array_equal(bits(resolve(s, 1)), bits(s))


# ---- 1. against the reference's own frames --------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("key,ss", [("default_96x54_d5", 2), ("default_96x54_d5", 3), ("synth256_96x80_d10", 2),
                                    ("synth256_96x80_d10", 4), ("two_mirrors_64x48_d50", 2),
                                    ("boxes_3_14_96x80_d12", 2)])
def test_ss_equals_resolved_golden_frame(gpu_ctx, golden, golden_frames, key, ss):
    """The goldens were rendered by the reference program itself, at the sample size."""
    m = golden["frames"][key]
    scene, cam = make_scene(m["scene"])
    gpu_ctx.upload(scene, cam)
    if m["scene"] == "synth256":
        assert gpu_ctx.scene_structures()["grid_cells"] > 0          # the grid kernel
    p = api.default_params(m["W"] // ss, m["H"] // ss, m["depth"])
    got, _ = gpu_ctx.render_ss(p, ss)
    assert_bit_identical(got, resolve(golden_frames[key], ss), f"{key} at ss={ss}")


# ---- 2. against the reference's md5s at full size -------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("key", ["default_500x504_d50", "default_1920x1080_d5"])
def test_ss_of_the_reference_configurations(gpu_ctx, golden, key):
    g = golden["md5"][key]
    scene, cam = make_scene(g["scene"])
    gpu_ctx.upload(scene, cam)
    sp = api.default_params(g["W"], g["H"], g["depth"])
    samples, st_s = gpu_ctx.render(sp)
    assert pixel_md5(gpu_ctx.format_txt()) == g["pixel_md5"]
    samples = samples.copy()
    got, st = gpu_ctx.render_ss(api.default_params(g["W"] // 2, g["H"] // 2, g["depth"]), 2)
    assert_bit_identical(got, resolve(samples, 2), f"{key} resolved at ss=2")
    assert st.rays == st_s.rays and st.rays_primary == g["W"] * g["H"]
    assert st.bands == [(0, g["W"] // 2)]


# ---- 3. ss = 1 is the plain frame ------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("scene", ["default", "two_mirrors", "synth256", "lattice:1:4"])
def test_ss1_is_the_plain_frame(gpu_ctx, scene):
    s, cam = make_scene(scene)
    gpu_ctx.upload(s, cam)
    p = api.default_params(160, 128, 12)
    img, st = gpu_ctx.render(p)
    img = img.copy()
    got, st1 = gpu_ctx.render_ss(p, 1)
    assert_bit_identical(got, img, f"{scene} ss=1")
    assert st1.rays == st.rays
    b8, st8 = gpu_ctx.render_rgb8(p)
    g8, st18 = gpu_ctx.render_ss_rgb8(p, 1)
    assert_bytes_equal(g8, b8, f"{scene} ss=1 RGB8")
    assert st18.rays == st8.rays


# ---- 4. odd shapes and untiled sample bands ---------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("w,h,ss,d", [(97, 61, 3, 8), (1, 1, 8, 50), (13, 7, 5, 12)])
def test_ss_odd_shapes(gpu_ctx, w, h, ss, d):
    """97 x 61 at ss = 3: 291 sample columns (not a multiple of the 4-column tile) and 183 rows; 1 x 1 at ss = 8; odd ss
    with scalar loads.  Against the plain render and the oracle at the sample size; then one-column bands."""
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    p = api.default_params(w, h, d)
    sp = sample_params(p, ss)
    samples, st_s = gpu_ctx.render(sp)
    want = resolve(samples, ss)
    got, st = gpu_ctx.render_ss(p, ss)
    assert_bit_identical(got, want, f"{w}x{h} ss={ss}")
    oracle, cnt = O.render(scene.flatten(), cam.export(), sp)
    assert_bit_identical(got, resolve(oracle, ss), f"{w}x{h} ss={ss} vs the oracle")
    assert (st.rays_primary, st.rays_shadow, st.rays_reflect) == (cnt["rays_primary"], cnt["rays_shadow"], cnt["rays_reflect"])
    assert st.rays == st_s.rays
    for x in sorted({0, w // 2, w - 1}):
        band, stb = gpu_ctx.render_ss(p, ss, x, x + 1)
        assert_bit_identical(band, want[x:x + 1], f"{w}x{h} ss={ss} column {x}")
        assert stb.bands == [(x, x + 1)]
        b8, _ = gpu_ctx.render_ss_rgb8(p, ss, x, x + 1)
        assert_bytes_equal(b8, q8(want[x:x + 1]), f"{w}x{h} ss={ss} column {x} RGB8")


# ---- 5. chunks, pinned and pageable, bands ----------------------------------------------------------------------------

GUARD = 4096


@gpu
def test_ss_chunked_pinned_and_pageable_destinations(gpu_ctx):
    """3840 x 2160 depth 50 at ss = 2 (a 7680 x 4320 sample frame).  [13, 1002) is 989 columns: its chunks start off the
    tile and, after the first, off the 16-byte alignment of the band."""
    scene, cam = make_scene("default")
    w, h, ss = 3840, 2160, 2
    p = api.default_params(w, h, 50)
    gpu_ctx.upload(scene, cam)
    samples, st_s = gpu_ctx.render(sample_params(p, ss))
    want = resolve(samples, ss)
    del samples
    want8 = q8(want)
    for x0, x1 in ((0, w), (13, 1002), (1, 3839)):
        n = (x1 - x0) * h * 3
        hbf, hb8 = api.HostBuffer(4 * n + GUARD), api.HostBuffer(n + GUARD)
        for kind, fbuf, bbuf in (("pinned", hbf.array(np.float32, (n + GUARD // 4,)), hb8.array(np.uint8, (n + GUARD,))),
                                 ("pageable", np.empty(n + GUARD // 4, np.float32), np.empty(n + GUARD, np.uint8))):
            fbuf.view(np.uint8)[:] = 0xAB
            _, st = gpu_ctx.render_ss(p, ss, x0, x1, out=fbuf[:n].reshape(x1 - x0, h, 3))
            assert st.gpu_launches > 4, "expected a chunked render"
            assert_bit_identical(fbuf[:n].reshape(x1 - x0, h, 3), want[x0:x1], f"[{x0},{x1}) {kind}")
            assert (fbuf[n:].view(np.uint8) == 0xAB).all(), f"[{x0},{x1}) {kind}: a guard byte was overwritten"
            if (x0, x1) == (0, w):
                assert st.rays == st_s.rays
            bbuf[:] = 0xAB
            gpu_ctx.render_ss_rgb8(p, ss, x0, x1, out=bbuf[:n].reshape(x1 - x0, h, 3))
            assert_bytes_equal(bbuf[:n].reshape(x1 - x0, h, 3), want8[x0:x1], f"[{x0},{x1}) {kind} RGB8")
            assert (bbuf[n:] == 0xAB).all(), f"[{x0},{x1}) {kind} RGB8: a guard byte was overwritten"
        del hbf, hb8
    # the device-only call is chunked too, and leaves the same frame
    st = gpu_ctx.render_ss_device(p, ss)
    assert st.gpu_launches > 4 and st.rays == st_s.rays
    got = gpu_ctx.download(np.empty((w, h, 3), np.float32))
    assert_bit_identical(got, want, "render_ss_device + download")


# ---- 6. scale and index range -----------------------------------------------------------------------------------------

def _chunk_starts(w, n_chunks=16):
    weights = [0, 1, 2, 4, 8, 12, 16, 20, 24, 28, 32, 36, 40, 42, 44, 45, 46]
    out = []
    for j in range(n_chunks + 1):
        c = w * weights[j] // weights[-1]
        if j < n_chunks and w % 4 == 0:
            c -= c % 4
        out.append(c)
    return out


@gpu
def test_ss4_at_8k(gpu_ctx):
    """synth256 7680 x 4320 depth 10 at ss = 4: 531 M samples in a 30720 x 17280 sample frame, which is never downloaded
    whole.  Column ranges, among them the first and last chunk boundaries, against the plain render of the matching
    sample columns."""
    scene, cam = make_scene("synth256")
    w, h, ss = 7680, 4320, 4
    p = api.default_params(w, h, 10)
    sp = sample_params(p, ss)
    gpu_ctx.upload(scene, cam)
    hb = api.HostBuffer(w * h * 12)
    got, st = gpu_ctx.render_ss(p, ss, out=hb.array(np.float32, (w, h, 3)))
    st_s = gpu_ctx.render_device(sp)
    assert st.rays == st_s.rays and st.rays_primary == sp.width * sp.height
    starts = _chunk_starts(w)
    ranges = [(0, 16), (starts[1] - 8, starts[1] + 8), (3836, 3850), (starts[-2] - 8, starts[-2] + 8), (w - 16, w)]
    for c0, c1 in ranges:
        samples, _ = gpu_ctx.render(sp, ss * c0, ss * c1)
        assert_bit_identical(got[c0:c1], resolve(samples, ss), f"synth256 8K ss=4 columns [{c0},{c1})")
    del got, hb


# ---- 7. the last render ----------------------------------------------------------------------------------------------

@gpu
def test_ss_frame_is_the_last_render(gpu_ctx, tmp_path):
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    p = api.default_params(160, 120, 20)
    samples, _ = gpu_ctx.render(sample_params(p, 2))
    plain, _ = gpu_ctx.render(p)
    plain = plain.copy()
    want = resolve(samples, 2)
    got, _ = gpu_ctx.render_ss_rgb8(p, 2)
    assert_bytes_equal(got, q8(want), "RGB8")
    assert_bit_identical(gpu_ctx.download(np.empty((160, 120, 3), np.float32)), want, "download")
    lib = _ffi.load()
    ptr, n = C.c_void_p(), C.c_size_t()
    assert lib.tcrt_device_frame(gpu_ctx._h, 0, C.byref(ptr), C.byref(n)) == 0
    assert n.value == 160 * 120 * 3
    torch = pytest.importorskip("torch")

    class _DeviceFrame:
        __cuda_array_interface__ = {"shape": (n.value,), "typestr": "<f4", "data": (ptr.value, False), "version": 3}

    dev = torch.as_tensor(_DeviceFrame(), device="cuda:0").cpu().numpy().reshape(160, 120, 3)
    assert_bit_identical(dev, want, "tcrt_device_frame")
    gpu_ctx.write_ppm(p, str(tmp_path / "ss.ppm"))
    ppm = (tmp_path / "ss.ppm").read_bytes()
    head = b"P6\n160 120\n255\n"
    assert ppm[:len(head)] == head
    image = np.frombuffer(ppm[len(head):], np.uint8).reshape(120, 160, 3)
    assert np.array_equal(image, q8(want).transpose(1, 0, 2)[::-1])
    gpu_ctx.write_txt(p, str(tmp_path / "ss.txt"))
    assert pixel_md5((tmp_path / "ss.txt").read_bytes()) == pixel_md5(O.format_txt(want))
    gpu_ctx.render(p)                                            # a plain frame restores the plain result
    assert_bit_identical(gpu_ctx.download(np.empty((160, 120, 3), np.float32)), plain, "plain frame afterwards")
    gpu_ctx.write_txt(p, str(tmp_path / "plain.txt"))
    assert pixel_md5((tmp_path / "plain.txt").read_bytes()) == pixel_md5(O.format_txt(plain))


# ---- 8. frames in flight ---------------------------------------------------------------------------------------------

@gpu
def test_ss_and_plain_async_frames_alternate(gpu_ctx):
    scene, cam = make_scene("default")
    w, h = 240, 150
    p = api.default_params(w, h, 12)
    gpu_ctx.upload(scene, cam)
    # (ss, format) per frame: supersampled and plain, float and RGB8
    kinds = [(2, "f"), (1, "f"), (3, "u8"), (2, "u8"), (1, "u8"), (3, "f"), (2, "f")]
    cams = []
    for i in range(len(kinds)):
        c = copy.copy(cam.export())
        c.eye[0] += 0.05 * i
        cams.append(c)
    want = []
    for (ss, fmt), c in zip(kinds, cams):
        gpu_ctx.set_camera(c)
        if fmt == "f":
            img, st = gpu_ctx.render_ss(p, ss) if ss > 1 else gpu_ctx.render(p)
        else:
            img, st = gpu_ctx.render_ss_rgb8(p, ss) if ss > 1 else gpu_ctx.render_rgb8(p)
        want.append((img.copy(), st.rays))
    hbs = [api.HostBuffer(w * h * (12 if fmt == "f" else 3)) for _, fmt in kinds]
    outs = [hb.array(np.float32 if fmt == "f" else np.uint8, (w, h, 3)) for hb, (_, fmt) in zip(hbs, kinds)]

    def submit(i):
        ss, fmt = kinds[i]
        if fmt == "f":
            return gpu_ctx.render_async_ss(p, ss, 0, w, outs[i]) if ss > 1 else gpu_ctx.render_async(p, out=outs[i])
        return gpu_ctx.render_async_ss_rgb8(p, ss, 0, w, outs[i]) if ss > 1 else gpu_ctx.render_async_rgb8(p, 0, w, outs[i])

    def check(i, st):
        if kinds[i][1] == "f":
            assert_bit_identical(outs[i], want[i][0], f"async frame {i} {kinds[i]}")
        else:
            assert_bytes_equal(outs[i], want[i][0], f"async frame {i} {kinds[i]}")
        assert st.rays == want[i][1]

    tickets = []
    for i, c in enumerate(cams):
        if len(tickets) == 2:
            j, t = tickets.pop(0)
            check(j, gpu_ctx.wait(t))
        gpu_ctx.set_camera(c)
        tickets.append((i, submit(i)))
        if len(tickets) == 2:
            for third in (lambda: gpu_ctx.render_async_ss(p, 2, 0, w, outs[0]),
                          lambda: gpu_ctx.render_async_ss_rgb8(p, 3, 0, w, outs[2])):
                with pytest.raises(api.TcrtError) as e:
                    third()
                assert e.value.code == _ffi.TCRT_ERR_INVALID
    for j, t in tickets:
        check(j, gpu_ctx.wait(t))
    # the last frame waited for was a supersampled float frame: it is the last render
    assert_bit_identical(gpu_ctx.download(np.empty((w, h, 3), np.float32)), want[-1][0], "download after async")
    gpu_ctx.set_camera(cam.export())


# ---- 9. error codes --------------------------------------------------------------------------------------------------

@gpu
def test_ss_error_codes(gpu_ctx):
    lib = _ffi.load()
    fresh = api.Context([0])
    p = api.default_params(8, 8, 2)
    with pytest.raises(api.TcrtError) as e:
        fresh.render_ss(p, 2)
    assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
    scene, cam = make_scene("default")
    fresh.upload(scene, cam)
    samples, _ = fresh.render(api.default_params(16, 16, 2))
    want = resolve(samples, 2)
    st = _ffi.TcrtStats()
    t = C.c_int(-1)
    buf = np.zeros(8 * 8 * 3, np.float32)
    buf8 = np.zeros(8 * 8 * 3, np.uint8)
    fdst, bdst = buf.ctypes.data_as(C.c_void_p), buf8.ctypes.data_as(C.c_void_p)
    wide = api.default_params((1 << 24) // 2 + 1, 1, 0)             # ss * width = 2^24 + 2
    tall = api.default_params(1, (1 << 22) + 1, 0)                   # ss * height = 2^24 + 4 at ss = 4
    cases = [(p, 0, _ffi.TCRT_ERR_INVALID), (p, -1, _ffi.TCRT_ERR_INVALID), (p, 9, _ffi.TCRT_ERR_UNSUPPORTED),
             (wide, 2, _ffi.TCRT_ERR_UNSUPPORTED), (tall, 4, _ffi.TCRT_ERR_UNSUPPORTED)]
    for q, ss, code in cases:
        assert lib.tcrt_render_columns_ss(fresh._h, C.byref(q), ss, 0, 1, fdst, C.byref(st)) == code, (ss, code)
        assert lib.tcrt_render_columns_ss(fresh._h, C.byref(q), ss, 0, 1, None, C.byref(st)) == code, (ss, code)
        assert lib.tcrt_render_columns_ss_rgb8(fresh._h, C.byref(q), ss, 0, 1, bdst, C.byref(st)) == code, (ss, code)
        assert lib.tcrt_render_async_ss(fresh._h, C.byref(q), ss, 0, 1, fdst, C.byref(t)) == code, (ss, code)
        assert lib.tcrt_render_async_ss_rgb8(fresh._h, C.byref(q), ss, 0, 1, bdst, C.byref(t)) == code, (ss, code)
        got, _ = fresh.render_ss(p, 2)                            # the context still renders correctly
        assert_bit_identical(got, want, f"after refusing ss={ss}")
    assert lib.tcrt_render_columns_ss_rgb8(fresh._h, C.byref(p), 2, 0, 8, None, C.byref(st)) == _ffi.TCRT_ERR_INVALID
    assert lib.tcrt_render_async_ss_rgb8(fresh._h, C.byref(p), 2, 0, 8, None, C.byref(t)) == _ffi.TCRT_ERR_INVALID
    for x0, x1 in ((3, 3), (5, 2), (-1, 4), (0, 9)):
        assert lib.tcrt_render_columns_ss(fresh._h, C.byref(p), 2, x0, x1, fdst, C.byref(st)) == _ffi.TCRT_ERR_INVALID
        assert lib.tcrt_render_async_ss(fresh._h, C.byref(p), 2, x0, x1, fdst, C.byref(t)) == _ffi.TCRT_ERR_INVALID
    assert (buf == 0).all() and (buf8 == 0).all()
    for ticket in (0, 1):                                    # nothing was queued by the refused calls
        with pytest.raises(api.TcrtError) as e:
            fresh.wait(ticket)
        assert e.value.code == _ffi.TCRT_ERR_INVALID
    got, _ = fresh.render_ss(p, 2)
    assert_bit_identical(got, want, "after the refusals")
    fresh.close()


# ---- 10. several GPUs in one context ---------------------------------------------------------------------------------

@gpu
def test_ss_multi_device_context_if_available(gpu_ctx):
    n = api.device_count()
    if n < 2:
        pytest.skip("one GPU visible")
    scene, cam = make_scene("default")
    p = api.default_params(1920, 1080, 5)
    gpu_ctx.upload(scene, cam)
    one, st1 = gpu_ctx.render_ss(p, 2)
    one = one.copy()
    one8, _ = gpu_ctx.render_ss_rgb8(p, 2)
    multi = api.Context(list(range(n)))
    multi.upload(scene, cam)
    for _ in range(2):                                    # the second frame is cut by the measured band times
        got, st = multi.render_ss(p, 2)
        assert st.n_devices == n and st.rays == st1.rays
        assert st.bands[0][0] == 0 and st.bands[-1][1] == 1920
        assert_bit_identical(got, one, f"ss=2 1080p on {n} GPUs")
        got8, _ = multi.render_ss_rgb8(p, 2)
        assert_bytes_equal(got8, one8, f"ss=2 1080p RGB8 on {n} GPUs")
    multi.close()


# ---- 11. C++ ---------------------------------------------------------------------------------------------------------

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
    RenderSettings rs;
    rs.width = 100; rs.height = 76; rs.max_depth = 50; rs.samples = 2;
    if (raytrace_main(scene, camera, rs, "raytracer_screen.txt")) return 1;
    GpuRayTracer rt;
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
def test_cpp_raytrace_main_with_samples(gpu_ctx, tmp_path):
    src = tmp_path / "render_ss.cpp"
    src.write_text(CPP_PROGRAM)
    libdir = os.path.join(ROOT, "tilecoderaytracer_b200")
    exe = tmp_path / "render_ss"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(ROOT, "include"), str(src),
                    "-L", libdir, "-ltcrt", f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    samples, _ = gpu_ctx.render(api.default_params(200, 152, 50))
    want = resolve(samples, 2)
    txt = (tmp_path / "raytracer_screen.txt").read_bytes()
    lines = [ln for ln in txt.split(b"\n") if ln.startswith(b"(")]
    assert b"\n".join(lines) + b"\n" == O.format_txt(want)
    got8 = np.fromfile(tmp_path / "frame.rgb8", dtype=np.uint8).reshape(100, 76, 3)
    assert_bytes_equal(got8, q8(want), "GpuRayTracer::renderRGB8 with samples = 2")
