"""GPU parity tests (-m gpu): the CUDA path, called through the C ABI, against
  * the oracle (CPU restatement pinned to the reference) on the same inputs — bit-exact,
  * the committed goldens made by the reference itself — bit-exact / md5-exact,
  * size-independent properties at the BASELINE.json sizes.

Stated tolerance of the north_star is <= 1 LSB per 8-bit channel on >= 99.9 % of pixels; the
bar enforced here is stricter: identical float bit patterns on every pixel (all arithmetic is
IEEE binary32, unfused, in the reference's order on both sides).
"""
import os
import tempfile

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api
from tilecoderaytracer_b200.partition import column_bands

from _util import assert_bit_identical, bits, make_scene, n_mismatch, parse_txt, pixel_md5, quant8

pytestmark = pytest.mark.gpu


def gpu_and_oracle(ctx, scene_name, w, h, depth, **kw):
    scene, cam = make_scene(scene_name)
    params = api.default_params(w, h, depth, **kw)
    ctx.upload(scene, cam)
    img, stats = ctx.render(params)
    want, cnt = O.render(scene.flatten(), cam.export(), params)
    return img, stats, want, cnt


def check_counters(stats, cnt):
    assert stats.rays_primary == cnt["rays_primary"]
    assert stats.rays_shadow == cnt["rays_shadow"]
    assert stats.rays_reflect == cnt["rays_reflect"]


# ---- against the oracle, same seeded inputs -------------------------------------------------------

@pytest.mark.parametrize("scene,w,h,d", [
    ("default", 500, 504, 50),        # BASELINE configs[0]
    ("default", 320, 180, 5),         # configs[1] scaled
    ("default", 97, 61, 0), ("default", 64, 48, 1), ("default", 64, 48, 200),
    ("synth1024", 160, 128, 50),      # configs[3] scaled
    ("synth256", 160, 128, 10),       # configs[4] scaled
    ("two_mirrors", 96, 80, 50),      # the reference's SCENE 2
])
def test_named_scenes_bit_exact(gpu_ctx, scene, w, h, d):
    img, stats, want, cnt = gpu_and_oracle(gpu_ctx, scene, w, h, d)
    assert_bit_identical(img, want, f"{scene} {w}x{h} d{d}")
    check_counters(stats, cnt)
    assert stats.gpu_launches == 1
    # the tolerance the north_star states, for the record
    assert (np.abs(quant8(img) - quant8(want)) <= 1).all(axis=-1).mean() >= 0.999


@pytest.mark.parametrize("seed,n", [(21, 12), (22, 40), (23, 90), (24, 200), (25, 600), (26, 33), (27, 1500), (28, 3)])
def test_random_scenes_bit_exact(gpu_ctx, seed, n):
    """Fuzz: every primitive type and ctor, lights of several types, textures, mirrors, diffuse-0."""
    img, stats, want, cnt = gpu_and_oracle(gpu_ctx, f"random:{seed}:{n}", 112, 80, 9)
    assert_bit_identical(img, want, f"random:{seed}:{n}")
    check_counters(stats, cnt)


@pytest.mark.parametrize("seed,n", [(1, 6), (2, 10), (3, 14), (4, 3), (5, 0), (6, 9), (7, 9), (8, 4)])
def test_axis_aligned_box_scenes_bit_exact(gpu_ctx, seed, n):
    """Fuzz of the box-cluster path: makeSceneBox boxes (stacked / abutting / duplicated: exact distance
    ties on coplanar faces go to the lower object index), lone axis-aligned rectangles of every sign
    combination, spheres and skewed planes in between, inside a closed room (up to 63 finite planes)."""
    img, stats, want, cnt = gpu_and_oracle(gpu_ctx, f"boxes:{seed}:{n}", 128, 96, 12)
    assert_bit_identical(img, want, f"boxes:{seed}:{n}")
    check_counters(stats, cnt)


@pytest.mark.parametrize("scene_name", ["default", "boxes:3:14", "boxes:7:9", "two_mirrors", "synth256", "synth1024"])
def test_axis_parallel_rays(gpu_ctx, scene_name):
    """A camera looking straight down +y with an axis-aligned screen: the centre column has D.x == 0
    and the centre row D.z == 0 exactly, and every mirror bounce off an axis-aligned face keeps such
    components zero.  Those rays bypass the box clusters' reciprocal (clu_wild) and hit den == 0 in the
    plane tests (SceneFinitePlane.cpp:96-97)."""
    scene, cam = make_scene(scene_name)
    c = cam.export()
    eye = (0.37, -6.2, 1.3)
    for k in range(3):
        c.eye[k] = eye[k]
        c.screen_origin[k] = eye[k] + (1.0 if k == 1 else 0.0)
        c.horizontal[k] = 1.0 if k == 0 else 0.0
        c.vertical[k] = 1.0 if k == 2 else 0.0
    p = api.default_params(96, 64, 12)
    gpu_ctx.upload_flat(scene.flatten(), c)
    img, stats = gpu_ctx.render(p)
    want, cnt = O.render(scene.flatten(), c, p)
    assert_bit_identical(img, want, f"{scene_name} axis-parallel camera")
    check_counters(stats, cnt)


def test_shared_reciprocal_division_is_ieee(gpu_ctx):
    """vector3d::normalize divides three components by one length (vector3d.h:57-74); the kernel
    shares the reciprocal between the three IEEE quotients.  2^31 random operand triples (zeros,
    denormals, |a| = b, exponents on both sides of the fast-path window) must agree with the
    division instruction sequence bit for bit."""
    for seed in (1, 2):
        assert gpu_ctx.selftest_div3(1 << 30, seed) == 0


@pytest.mark.parametrize("scene,w,h,d", [
    ("boxes:11:9", 136, 104, 15), ("boxes:12:4", 100, 60, 50), ("random:15:90", 136, 104, 25),
    ("random:16:7", 97, 61, 50), ("synth1024", 136, 104, 3), ("synth256", 97, 61, 30),
])
def test_more_scenes_tiled_and_untiled_sizes(gpu_ctx, scene, w, h, d):
    """Frame sizes that are (136x104) and are not (100x60, 97x61) multiples of the 4x8 pixel tile, deep and
    shallow recursion caps."""
    img, stats, want, cnt = gpu_and_oracle(gpu_ctx, scene, w, h, d)
    assert_bit_identical(img, want, f"{scene} {w}x{h} d{d}")
    check_counters(stats, cnt)


def test_switches_shadows_reflections(gpu_ctx):
    for kw in ({"shadows": False}, {"reflections": False}, {"shadows": False, "reflections": False}):
        img, stats, want, cnt = gpu_and_oracle(gpu_ctx, "default", 120, 90, 7, **kw)
        assert_bit_identical(img, want, str(kw))
        check_counters(stats, cnt)


def test_handmade_scene_edge_cases(gpu_ctx):
    """Camera inside a sphere (negative distance wins, SceneSphere.cpp:139), a plane light, a
    textured finite plane, coincident spheres (index tie-break, RayTracer.cpp:77), no lights."""
    cam = api.Camera()
    eye = np.array(cam.export().eye[:], np.float32)
    for variant in range(4):
        s = api.Scene()
        if variant != 3:
            s.addFinitePlaneCorners((2, 2, 9), (2, 2.5, 9), (2.5, 2, 9)).setAsLightSource(0.9)
            s.addSphere((-6, 0, 8), .2).setAsLightSource(0.5).setColor(1, .5, .25)
        if variant == 0:
            s.addSphere(tuple(eye), 3.0).setColor(.2, .4, .9)            # we are inside this one
        s.addSphere((0, 0, 1), 1.0).setColor(1, 0, 0).setReflectiveFactor(.7)
        s.addSphere((0, 0, 1), 1.0).setColor(0, 1, 0)                   # coincident: the red one must win
        s.addInfinitePlane((0, 0, 0), (0, 0, 1), (1, 0, 0)).setCheckerBoard((1, 1, 0), (0, 0, 1), 1.5, .7)
        s.addFinitePlaneAxes((-1, 3, 0), (0, -1, 0), (1, 0, 0), 2.5, 3.0).setCheckerBoard((1, 1, 1), (.1, .1, .1), .5, .5) \
            .setReflectiveFactor(.4).setDiffuseFactor(0.0)
        if variant == 2:
            for o in s.makeSceneBox((-3, -3, 0), (1, 1, 2)):
                o.setColor(.6, .3, .1).setSpecularFactor(.3)
        params = api.default_params(140, 100, 6)
        gpu_ctx.upload(s, cam)
        img, stats = gpu_ctx.render(params)
        want, cnt = O.render(s.flatten(), cam.export(), params)
        assert_bit_identical(img, want, f"handmade variant {variant}")
        check_counters(stats, cnt)


def test_empty_scene_and_tiny_images(gpu_ctx):
    cam = api.Camera()
    gpu_ctx.upload(api.Scene(), cam)
    img, stats = gpu_ctx.render(api.default_params(33, 17, 4))
    assert np.all(img == np.float32(0.75)) and stats.rays == 33 * 17
    scene, cam = make_scene("default")
    gpu_ctx.upload(scene, cam)
    for w, h in [(1, 1), (1, 37), (37, 1), (2, 3)]:
        p = api.default_params(w, h, 50)
        img, stats = gpu_ctx.render(p)
        want, _ = O.render(scene.flatten(), cam.export(), p)
        assert_bit_identical(img, want, f"{w}x{h}")
        assert stats.rays_primary == w * h


def test_maximum_object_count(gpu_ctx):
    """3999 objects = the most Scene::addObject accepts (Scene.cpp:470-479)."""
    cam = api.Camera()
    s = api.Scene()
    s.addSphere((2, -3, 9), .2).setAsLightSource(1.0)
    s.addInfinitePlane((0, 0, 0), (0, 0, 1), (1, 0, 0)).setCheckerBoard((1, 1, 1), (0, 0, 0), 3, 3)
    k = 0
    while s.getObjectCount() < 3999:
        i, j, l = k % 20, (k // 20) % 20, k // 400
        s.addSphere((-2 + .45 * i, .45 * j, .2 + .45 * l), .2).setColor((i % 3) / 2, (j % 3) / 2, (l % 3) / 2) \
            .setReflectiveFactor(.5 if k % 7 == 0 else 0.0)
        k += 1
    assert s.getObjectCount() == 3999
    gpu_ctx.upload(s, cam)
    p = api.default_params(64, 48, 4)
    img, stats = gpu_ctx.render(p)
    want, cnt = O.render(s.flatten(), cam.export(), p)
    assert_bit_identical(img, want, "3999 objects")
    check_counters(stats, cnt)


# ---- against the committed goldens (made by the reference itself) -------------------------------------

def test_golden_frames_bit_exact(gpu_ctx, golden, golden_frames):
    for key, m in golden["frames"].items():
        scene, cam = make_scene(m["scene"])
        gpu_ctx.upload(scene, cam)
        img, _ = gpu_ctx.render(api.default_params(m["W"], m["H"], m["depth"]))
        assert_bit_identical(img, golden_frames[key], key)


@pytest.mark.parametrize("key", ["default_500x504_d50", "default_1920x1080_d5", "synth1024_500x504_d50",
                                 "synth256_500x504_d10", "two_mirrors_500x504_d50", "random_4_80_200x160_d8",
                                 "default_3840x2160_d50"])
def test_txt_md5_matches_reference_file(gpu_ctx, golden, key):
    """Render + GPU .txt formatter + file writer; md5 of the pixel lines equals the reference
    program's.  default_500x504_d50 is the program exactly as checked in (rt_asis)."""
    g = golden["md5"][key]
    scene, cam = make_scene(g["scene"])
    gpu_ctx.upload(scene, cam)
    p = api.default_params(g["W"], g["H"], g["depth"])
    gpu_ctx.render_device(p)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "raytracer_screen.txt")
        gpu_ctx.write_txt(p, path, run_time_s=0.25)
        txt = open(path, "rb").read()
    body = txt[txt.index(b"("):]
    assert len(body) == g["pixel_bytes"]
    assert pixel_md5(txt) == g["pixel_md5"]
    head = txt[:txt.index(b"(")].decode().splitlines()
    assert head[0] == "OSX Awesome Picture" and head[1] == f"Horizontal_Resolution:{g['W']}."
    assert head[7] == "Run_Time:0.250000." and len(head) == 10


# ---- the writer on arbitrary floats ------------------------------------------------------------------

def test_writer_known_answers(gpu_ctx):
    """main_test()'s gradient (RayTracer.cpp:1412-1444) and hand-picked values through the GPU
    formatter vs glibc's "%f" (oracle) and Python's correctly rounded '%f'."""
    w, h = 500, 504
    i = np.arange(w, dtype=np.float32)[:, None] / np.float32(w)
    j = np.arange(h, dtype=np.float32)[None, :] / np.float32(h)
    px = np.stack([np.broadcast_to(i, (w, h)), np.broadcast_to(j, (w, h)), np.full((w, h), .5, np.float32)], -1)
    got = gpu_ctx.format_pixels(px)
    assert got == O.format_txt(px)
    assert got.startswith(b"(0.000000, 0.000000, 0.500000)\n(0.000000, 0.001984, 0.500000)\n")
    assert len(got) == w * h * 31
    special = np.array([
        [0.0, 1.0, 9.999999], [9.9999995, 0.0000005, 0.0000015], [0.0000025, 0.5, 0.125],
        [1e-7, 4.9999997e-7, 5.0000003e-7], [1e-45, 1.17549435e-38, 2.5e-7],
        [10.0, 123456.789, 16777216.0], [-0.0, -1.5, -0.0000004], [3.4028235e38, 1e20, 65535.0],
        [np.inf, -np.inf, np.nan], [2.684511, 4.26, 0.75],
    ], dtype=np.float32)
    got = gpu_ctx.format_pixels(special)
    assert got == O.format_txt(special)
    lines = got.decode().splitlines()
    for row, line in zip(special, lines):
        if np.isfinite(row).all():
            assert line == "(%f, %f, %f)" % tuple(float(v) for v in row)
    assert lines[8] == "(inf, -inf, nan)"


def test_writer_random_floats_fixed_and_general_paths(gpu_ctx):
    rng = np.random.default_rng(1234)
    # fixed path: all in [0, 10)
    a = rng.random((50000, 3), dtype=np.float32) * np.float32(9.99)
    a[::7] *= np.float32(1e-4)
    assert gpu_ctx.format_pixels(a) == O.format_txt(a)
    # exact ties of the 6th decimal: k + 0.5 micro-units that are representable
    ties = (np.arange(1, 3001, dtype=np.float64) * 2 + 1) * 2.0 ** -21   # odd / 2^21
    t32 = ties.astype(np.float32).reshape(-1, 3)
    assert gpu_ctx.format_pixels(t32) == O.format_txt(t32)
    # general path: random bit patterns (any exponent, sign, subnormals), no NaN payload issues
    raw = rng.integers(0, 2 ** 32, size=(30000, 3), dtype=np.uint64).astype(np.uint32)
    b = raw.view(np.float32)
    b = np.where(np.isnan(b), np.float32(1.0), b)
    got = gpu_ctx.format_pixels(b)
    assert got == O.format_txt(b)
    # mixed: mostly fixed with a few long lines
    c = a.copy()
    c[123, 1] = 10.5
    c[40000, 0] = -3.0
    assert gpu_ctx.format_pixels(c) == O.format_txt(c)


# ---- properties at the BASELINE sizes -------------------------------------------------------------------

def sampled_columns_match(ctx, scene_name, w, h, d, stride):
    scene, cam = make_scene(scene_name)
    ctx.upload(scene, cam)
    p = api.default_params(w, h, d)
    img, stats = ctx.render(p)
    want, _ = O.render(scene.flatten(), cam.export(), p, 0, w, stride)
    assert_bit_identical(img[0:w:stride], want, f"{scene_name} {w}x{h} sampled columns")
    return img, stats, p


def test_1080p_depth5_sampled_parity_and_band_stitching(gpu_ctx):
    """configs[1]: every 16th column against the oracle; then the same image rendered as 1, 3 and
    8 bands must be the same bits (the result of a pixel does not depend on the partition)."""
    img, stats, p = sampled_columns_match(gpu_ctx, "default", 1920, 1080, 5, 16)
    for n in (3, 8):
        parts = []
        rays = 0
        for x0, x1 in column_bands(1920, n):
            band, st = gpu_ctx.render(p, x0, x1)
            parts.append(band)
            rays += st.rays
        assert np.array_equal(bits(np.concatenate(parts, 0)), bits(img))
        assert rays == stats.rays
    again, st2 = gpu_ctx.render(p)
    assert np.array_equal(bits(again), bits(img)) and st2.rays == stats.rays     # idempotent


def test_4k_depth50_sampled_parity_and_txt_round_trip(gpu_ctx):
    """configs[2] on one GPU: sampled columns vs oracle; .txt lines parse back to the floats
    (6 decimals) and every line is 31 bytes."""
    img, stats, p = sampled_columns_match(gpu_ctx, "default", 3840, 2160, 50, 128)
    assert stats.rays_primary == 3840 * 2160
    n = gpu_ctx.txt_size()
    assert n == 3840 * 2160 * 31
    txt = gpu_ctx.format_txt()
    assert txt[30:31] == b"\n" and txt[-1:] == b"\n"
    sub = txt[: 31 * 2160 * 4]
    vals = parse_txt(sub).reshape(4, 2160, 3)
    assert np.abs(vals - img[:4].astype(np.float64)).max() <= 0.5e-6 + 1e-12


def test_synth1024_4k_sampled_parity(gpu_ctx):
    """configs[3]: 1027 objects at 3840x2160, every 256th column against the oracle."""
    sampled_columns_match(gpu_ctx, "synth1024", 3840, 2160, 50, 256)


def test_synth256_8k_sampled_parity(gpu_ctx):
    """configs[4]: 259 objects at 7680x4320 depth 10, every 512th column against the oracle."""
    img, stats, p = sampled_columns_match(gpu_ctx, "synth256", 7680, 4320, 10, 512)
    assert img.shape == (7680, 4320, 3) and np.isfinite(img).all() and img.min() >= 0


# ---- error behaviour of the boundary -------------------------------------------------------------------

def test_error_codes(gpu_ctx, tmp_path):
    fresh = api.Context([0])
    p = api.default_params(8, 8, 2)
    with pytest.raises(api.TcrtError) as e:
        fresh.render(p)
    assert e.value.code == _ffi.TCRT_ERR_NO_SCENE
    scene, cam = make_scene("default")
    fresh.upload(scene, cam)
    with pytest.raises(api.TcrtError) as e:
        fresh.txt_size()
    assert e.value.code == _ffi.TCRT_ERR_NO_FRAME
    for bad in (api.default_params(0, 8, 2), api.default_params(8, -1, 2), api.default_params(8, 8, -1)):
        with pytest.raises(api.TcrtError) as e:
            fresh.render_device(bad, 0, 1)
        assert e.value.code == _ffi.TCRT_ERR_INVALID
    with pytest.raises(api.TcrtError) as e:
        fresh.render_device(api.default_params(8, 8, 255))
    assert e.value.code == _ffi.TCRT_ERR_UNSUPPORTED
    with pytest.raises(api.TcrtError) as e:
        fresh.render_device(p, 3, 3)
    assert e.value.code == _ffi.TCRT_ERR_INVALID
    fresh.render_device(p, 2, 6)
    with pytest.raises(api.TcrtError) as e:
        fresh.write_txt(p, str(tmp_path / "should_not_exist.txt"))       # band, not the whole image
    assert e.value.code == _ffi.TCRT_ERR_INVALID
    assert not (tmp_path / "should_not_exist.txt").exists()
    fresh.render_device(p)
    with pytest.raises(api.TcrtError) as e:
        fresh.write_txt(p, str(tmp_path / "nonexistent_dir" / "x" / "raytracer_screen.txt"))
    assert e.value.code == _ffi.TCRT_ERR_IO
    with pytest.raises(api.TcrtError) as e:
        api.Context([99])
    assert e.value.code == _ffi.TCRT_ERR_NO_DEVICE
    fresh.close()


def test_cost_balanced_bands_on_gpu(gpu_ctx):
    """tcrt_balance_columns: tiles the frame and evens out the per-band ray counts of
    the mirror-heavy scene compared with equal widths; stitched bands are the same bits as one render."""
    scene, cam = make_scene("synth256")
    p = api.default_params(512, 288, 10)
    gpu_ctx.upload(scene, cam)
    full, st = gpu_ctx.render(p)
    for n in (2, 4, 8):
        bands = gpu_ctx.balance_columns(p, n)
        assert bands[0][0] == 0 and bands[-1][1] == 512 and all(a[1] == b[0] for a, b in zip(bands, bands[1:]))
        rays_bal, rays_eq = [], []
        parts = []
        for x0, x1 in bands:
            img, s = gpu_ctx.render(p, x0, x1)
            parts.append(img)
            rays_bal.append(s.rays)
        assert np.array_equal(bits(np.concatenate(parts, axis=0)), bits(full))
        for x0, x1 in column_bands(512, n):
            rays_eq.append(gpu_ctx.render_device(p, x0, x1).rays)
        assert sum(rays_bal) == sum(rays_eq) == st.rays
        assert max(rays_bal) <= max(rays_eq) * 1.02
        assert max(rays_bal) <= 1.25 * st.rays / n


def test_image_outputs_and_camera_update(gpu_ctx, tmp_path):
    """SURVEY §8f rows: PPM / raw-float outputs of a frame and tcrt_set_camera (multi-frame mode)."""
    scene, cam = make_scene("default")
    p = api.default_params(96, 64, 6)
    gpu_ctx.upload(scene, cam)
    img, _ = gpu_ctx.render(p)
    gpu_ctx.write_ppm(p, str(tmp_path / "a.ppm"))
    raw = (tmp_path / "a.ppm").read_bytes()
    head = b"P6\n96 64\n255\n"
    assert raw.startswith(head) and len(raw) == len(head) + 96 * 64 * 3
    got = np.frombuffer(raw[len(head):], dtype=np.uint8).reshape(64, 96, 3)
    want = np.transpose(quant8(img), (1, 0, 2))[::-1].astype(np.uint8)
    assert np.array_equal(got, want)
    # a frame that is not a multiple of the 32x32 transposition tile
    p2 = api.default_params(97, 61, 4)
    img2, _ = gpu_ctx.render(p2)
    gpu_ctx.write_ppm(p2, str(tmp_path / "b.ppm"))
    raw2 = (tmp_path / "b.ppm").read_bytes()
    head2 = b"P6\n97 61\n255\n"
    got2 = np.frombuffer(raw2[len(head2):], dtype=np.uint8).reshape(61, 97, 3)
    assert np.array_equal(got2, np.transpose(quant8(img2), (1, 0, 2))[::-1].astype(np.uint8))
    img, _ = gpu_ctx.render(p)
    gpu_ctx.write_bin(p, str(tmp_path / "a.bin"))
    rawb = (tmp_path / "a.bin").read_bytes()
    assert rawb[:8] == b"TCRTBIN1" and np.frombuffer(rawb[8:16], dtype=np.int32).tolist() == [96, 64]
    assert np.array_equal(np.frombuffer(rawb[32:], dtype=np.float32).view(np.uint32), bits(img).ravel())
    # a moved camera without re-uploading the scene == uploading with that camera
    cam2 = cam.export()
    cam2.eye[0] += 0.25
    cam2.eye[2] += 0.1
    gpu_ctx.set_camera(cam2)
    moved, _ = gpu_ctx.render(p)
    assert n_mismatch(moved, img) > 0
    gpu_ctx.upload_flat(scene.flatten(), cam2)
    again, _ = gpu_ctx.render(p)
    assert_bit_identical(moved, again, "set_camera vs upload")
    want2, _ = O.render(scene.flatten(), cam2, p)
    assert_bit_identical(moved, want2, "moved camera vs oracle")


def test_multi_device_context_if_available(gpu_ctx):
    """In-process band split over every visible GPU: same bits as one GPU."""
    n = api.device_count()
    if n < 2:
        pytest.skip("one GPU visible")
    scene, cam = make_scene("default")
    p = api.default_params(640, 360, 8)
    gpu_ctx.upload(scene, cam)
    one, st1 = gpu_ctx.render(p)
    multi = api.Context(list(range(n)))
    multi.upload(scene, cam)
    img, st = multi.render(p)
    assert st.n_devices == n      # bands: the cost-balanced cut
    assert st.bands[0][0] == 0 and st.bands[-1][1] == 640 and all(a[1] == b[0] for a, b in zip(st.bands, st.bands[1:]))
    assert np.array_equal(bits(img), bits(one)) and st.rays == st1.rays
    multi.render_device(p)
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "a.txt")
        multi.write_txt(p, path)
        gpu_ctx.render_device(p)
        gpu_ctx.write_txt(p, os.path.join(td, "b.txt"))
        assert open(path, "rb").read() == open(os.path.join(td, "b.txt"), "rb").read()
    multi.close()


def test_cpp_host_program_is_a_drop_in(golden, tmp_path):
    """examples/raytrace_main.cpp: the reference's main()/raytrace_main() flow written against the
    drop-in C++ headers, linked with libtcrt.so.  Its raytracer_screen.txt must carry the same pixel
    lines as the reference program's (rt_asis) and the same header layout."""
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    libdir = os.path.join(root, "tilecoderaytracer_b200")
    exe = tmp_path / "raytrace_main"
    subprocess.run(["g++", "-std=c++17", "-O2", "-ffp-contract=off", "-I", os.path.join(root, "include"),
                    os.path.join(root, "examples", "raytrace_main.cpp"), "-L", libdir, "-ltcrt",
                    f"-Wl,-rpath,{libdir}", "-o", str(exe)], check=True)
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    txt = (tmp_path / "raytracer_screen.txt").read_bytes()
    assert pixel_md5(txt) == golden["asis"]["rt_asis"]["pixel_md5"]
    head = txt[:txt.index(b"(")].decode().splitlines()
    want = golden["asis"]["rt_asis"]["header_lines"]
    strip = lambda ls: [l for l in ls if not l.startswith(("Run_Time", "us/pixel"))]
    assert strip(head) == strip(want) and len(head) == len(want)
    # SCENE 2 through the same program
    r = subprocess.run([str(exe), "2"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    txt = (tmp_path / "raytracer_screen.txt").read_bytes()
    assert pixel_md5(txt) == golden["md5"]["two_mirrors_500x504_d50"]["pixel_md5"]


def test_bench_dump_outputs_are_the_timed_frame(golden, tmp_path):
    """bench.py --dump-outputs: on the reference's own configuration (small enough to be written whole) the dumped
    frame carries the reference program's pixel lines, and the dumped counters are that frame's rays."""
    import json
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--workload", "default_500x504_d50", "--steps", "2",
                        "--warmup", "1", "--quick", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout)
    assert line["steps"] == 2
    img, cols, rays = (np.load(out / f) for f in ("image.npy", "image_columns.npy", "rays.npy"))
    assert img.dtype == np.float32 and img.shape == (500, 504, 3)
    assert np.array_equal(cols, np.arange(500))
    assert pixel_md5(O.format_txt(img)) == golden["md5"]["default_500x504_d50"]["pixel_md5"]
    assert rays.tolist() == [252000, 963640, 230689] and line["rays_per_frame"] == rays.sum()


# ---- round 2: the sphere BVH that collapses into one leaf, text scenes ---------------------------------

def _render_vs_oracle(ctx, s, cam, w=112, h=80, d=8, what=""):
    p = api.default_params(w, h, d)
    ctx.upload(s, cam)
    img, stats = ctx.render(p)
    want, cnt = O.render(s.flatten(), cam.export(), p)
    assert_bit_identical(img, want, what)
    check_counters(stats, cnt)


def _lights_and_ground(s):
    s.addSphere((-2, -6, 12), .15).setAsLightSource(.75)
    s.addSphere((8, 2, 10), .15).setAsLightSource(1.0)
    s.addInfinitePlane((0, 0, 0), (0, 0, 1), (1, 0, 0)).setCheckerBoard((1, 1, 1), (0, 0, 0), 3, 3) \
        .setReflectiveFactor(.5).setDiffuseFactor(.5)


def test_named_scenes_take_their_intended_structures(gpu_ctx):
    """default: box clusters, no BVH; synth256 / synth1024: sphere grid (+ BVH for far origins); SCENE 2: sphere BVH only (its
    radius-10 sphere rules a grid out); a random scene with many finite planes: their BVH."""
    want = {"default": dict(grid_cells=0, bvh_spheres=0, clusters=4, cluster_rects=24), "synth256": dict(bvh_spheres=256), "synth1024": dict(bvh_spheres=1024),
            "two_mirrors": dict(grid_cells=0), "random:27:1500": dict(grid_cells=0)}
    for name, exp in want.items():
        scene, cam = make_scene(name)
        gpu_ctx.upload(scene, cam)
        got = gpu_ctx.scene_structures()
        for k, v in exp.items():
            assert got[k] == v, (name, got)
        if name.startswith("synth"):
            assert got["grid_cells"] > 0, (name, got)
        if name in ("two_mirrors", "random:27:1500"):
            assert got["bvh_spheres"] > 0 or got["bvh_finite"] > 0, (name, got)


def test_sphere_bvh_collapsing_into_one_leaf(gpu_ctx):
    """>= 24 non-light spheres ask for a BVH, but after the exclusions (16 tiny spheres stay linear) only
    8 coincident ones are left and SAH keeps them in ONE leaf: there are no nodes, the kernel without a
    sphere BVH runs and must stage and sweep all 24 (tcrt_upload_scene once sized shared memory as if
    8 of them were BVH-covered)."""
    cam = api.Camera()
    s = api.Scene()
    _lights_and_ground(s)
    for k in range(16):
        s.addSphere((-1.5 + .4 * (k % 4), -1.0 + .4 * (k // 4), .3 + .05 * k), .02 + .001 * k) \
            .setColor(1, k / 16, 0).setReflectiveFactor(.3 if k % 3 == 0 else 0.0)
    for k in range(8):
        s.addSphere((0.5, 0.5, 1.0), 1.0).setColor(k / 8, 1 - k / 8, .5).setReflectiveFactor(.5 if k == 0 else 0.0)
    _render_vs_oracle(gpu_ctx, s, cam, what="24 spheres: 16 tiny + 8 coincident")


@pytest.mark.parametrize("n_zero,n_real", [(30, 3), (40, 0), (26, 6), (5, 30)])
def test_zero_radius_spheres(gpu_ctx, n_zero, n_real):
    """Zero-radius spheres never enter the BVH (they would make the per-ray fattening infinite); with few
    real spheres left the tree is a single leaf or empty."""
    cam = api.Camera()
    s = api.Scene()
    _lights_and_ground(s)
    for k in range(n_zero):
        s.addSphere((-2 + .13 * k, -1 + .07 * k, .5 + .02 * k), 0.0).setColor(1, 0, 1)
    for k in range(n_real):
        s.addSphere((-1 + .9 * (k % 6), .5 * (k // 6), .6 + .1 * (k % 3)), .45).setColor(.2, .3 + .1 * (k % 5), 1) \
            .setReflectiveFactor(.6 if k % 2 else 0.0)
    _render_vs_oracle(gpu_ctx, s, cam, what=f"{n_zero} zero-radius + {n_real} spheres")


def test_text_scene_renders_like_the_oracle(gpu_ctx):
    """SURVEY §8f row 3: scenes/default.scene through tcrt_hscene_load_text, rendered on the GPU, against the
    oracle on the same flattened arrays AND against the built-in Scene::initialize() frame."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cam = api.Camera()
    s = api.Scene().load_text(os.path.join(root, "scenes", "default.scene"), cam)
    p = api.default_params(200, 152, 50)
    gpu_ctx.upload(s, cam)
    img, stats = gpu_ctx.render(p)
    want, cnt = O.render(s.flatten(), cam.export(), p)
    assert_bit_identical(img, want, "default.scene vs oracle")
    check_counters(stats, cnt)
    scene2, cam2 = make_scene("default")
    gpu_ctx.upload(scene2, cam2)
    img2, _ = gpu_ctx.render(p)
    assert_bit_identical(img, img2, "default.scene vs Scene::initialize()")


# ---- round 2: asynchronous frames, the pipelined writer, the scene cache -------------------------------------

def test_async_frames_equal_synchronous_frames(gpu_ctx):
    """tcrt_render_async / tcrt_wait: two frames in flight with different cameras, each into its own pinned
    buffer, are the frames the synchronous call renders; a third submit is refused until one is waited for."""
    import copy

    scene, cam = make_scene("default")
    p = api.default_params(320, 200, 12)
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
    bufs = [api.HostBuffer(320 * 200 * 12) for _ in range(2)]
    outs = [b.array(np.float32, (320, 200, 3)) for b in bufs]
    tickets = []
    for i, c in enumerate(cams):
        if len(tickets) == 2:
            j, t = tickets.pop(0)
            st = gpu_ctx.wait(t)
            assert np.array_equal(bits(outs[j % 2]), bits(want[j][0])) and st.rays == want[j][1]
        gpu_ctx.set_camera(c)
        tickets.append((i, gpu_ctx.render_async(p, out=outs[i % 2])))
    with pytest.raises(api.TcrtError):
        gpu_ctx.render_async(p, out=outs[0])          # two already in flight
    for j, t in tickets:
        st = gpu_ctx.wait(t)
        assert np.array_equal(bits(outs[j % 2]), bits(want[j][0])) and st.rays == want[j][1]
    with pytest.raises(api.TcrtError):
        gpu_ctx.wait(0)                                # nothing pending any more
    # the frame last waited for is "the last render" of the synchronous calls
    got = np.empty((320, 200, 3), np.float32)
    gpu_ctx.download(got)
    assert np.array_equal(bits(got), bits(want[-1][0]))
    gpu_ctx.set_camera(cam.export())


def test_writer_falls_back_to_the_general_layout(gpu_ctx, tmp_path):
    """A light of intensity 12 seen directly gives channels >= 10: pixel lines longer than 31 bytes.  The
    pipelined fixed-width writer must notice and produce the general layout: the file equals glibc's."""
    cam = api.Camera()
    s = api.Scene()
    s.addSphere((-2, -2, 2.0), .8).setAsLightSource(12.0)
    s.addInfinitePlane((0, 0, 0), (0, 0, 1), (1, 0, 0)).setCheckerBoard((1, 1, 1), (0, 0, 0), 3, 3)
    s.addSphere((0, 0, 1), 1.0).setColor(1, 0, 0).setReflectiveFactor(.7)
    p = api.default_params(160, 120, 6)
    gpu_ctx.upload(s, cam)
    img, _ = gpu_ctx.render(p)
    assert img.max() >= 10.0
    path = str(tmp_path / "raytracer_screen.txt")
    gpu_ctx.write_txt(p, path, 0.5)
    txt = open(path, "rb").read()
    assert txt == api.txt_header(p, 0.5) + O.format_txt(img)
    with pytest.raises(api.TcrtError) as e:
        api.txt_create(p, path, 0.5)
        gpu_ctx.write_txt_band(p, path, 0.5)
    assert e.value.code == _ffi.TCRT_ERR_UNSUPPORTED


def test_bands_written_into_one_file(gpu_ctx, tmp_path):
    """tcrt_txt_create + tcrt_write_txt_band (what one rank per GPU does): bands written in any order give the
    file tcrt_write_txt gives."""
    scene, cam = make_scene("default")
    p = api.default_params(640, 360, 8)
    gpu_ctx.upload(scene, cam)
    gpu_ctx.render_device(p)
    whole = str(tmp_path / "whole.txt")
    gpu_ctx.write_txt(p, whole, 1.25)
    parts = str(tmp_path / "parts.txt")
    api.txt_create(p, parts, 1.25)
    for x0, x1 in reversed(column_bands(640, 5)):
        gpu_ctx.render_device(p, x0, x1)
        gpu_ctx.write_txt_band(p, parts, 1.25)
    assert open(parts, "rb").read() == open(whole, "rb").read()
    # a file that tcrt_txt_create did not make for these params is refused
    with pytest.raises(api.TcrtError) as e:
        gpu_ctx.write_txt_band(p, parts, 12345.0)      # longer header -> other size
    assert e.value.code == _ffi.TCRT_ERR_INVALID


def test_scene_cache_sees_every_change(gpu_ctx):
    """tcrt_upload_scene skips the rebuild for a bit-identical scene; any change must rebuild."""
    cam = api.Camera()
    p = api.default_params(96, 72, 6)

    def build(shift, color):
        s = api.Scene()
        _lights_and_ground(s)
        for k in range(30):
            s.addSphere((-1 + .5 * (k % 6) + shift, .5 * (k // 6), .6), .22).setColor(color, .5, 1 - color) \
                .setReflectiveFactor(.5 if k % 2 else 0.0)
        return s

    for shift, color in [(0.0, .2), (0.0, .2), (0.25, .2), (0.25, .9), (0.0, .2)]:
        s = build(shift, color)
        gpu_ctx.upload(s, cam)
        img, stats = gpu_ctx.render(p)
        want, cnt = O.render(s.flatten(), cam.export(), p)
        assert_bit_identical(img, want, f"shift {shift} color {color}")
        check_counters(stats, cnt)


# ---- round 2: the uniform grid over lattice-like sphere scenes (tcrt_render_grid.cu) ---------------------------------------

def _lattice(s, nx, ny, nz, spacing, radius, jitter=0.0, rvar=0.0, seed=1):
    rng = np.random.default_rng(seed)
    for k in range(nz):
        for j in range(ny):
            for i in range(nx):
                c = np.array([-3 + spacing * i, -1 + spacing * j, radius + .05 + spacing * k]) + jitter * (rng.random(3) - .5)
                r = radius * (1 + rvar * (rng.random() - .5))
                s.addSphere(tuple(float(x) for x in c), float(r)).setColor(*(float(x) for x in rng.random(3))) \
                    .setReflectiveFactor(float(.9 if (i + j + k) % 2 else 0.0)).setDiffuseFactor(.3)


@pytest.mark.parametrize("case", ["far_camera", "inside_sphere", "jittered", "row_of_200", "dense_small", "three_lights"])
def test_sphere_grid_edge_cases(gpu_ctx, case):
    """Scenes whose spheres go into the uniform grid, rendered bit for bit like the oracle: a camera 600 units away
    (every primary ray's fattening exceeds the grid's margin: BVH fallback, and far ground hits send far shadow and
    mirror rays), a camera inside a sphere of the lattice (negative distances win), jittered positions and radii
    (spheres registered in several cells), a row of 200 spheres (more cells than the 64 per axis the grid allows),
    a dense lattice of small spheres, and three lights (three shadow passes per bounce)."""
    cam = api.Camera()
    c = cam.export()
    s = api.Scene()
    _lights_and_ground(s)
    w, h, d = 128, 96, 8
    if case == "far_camera":
        _lattice(s, 6, 6, 3, 1.8, .75)
        for k in range(3):      # move eye and screen 600 units back along the viewing direction (0.62, 0.78, 0.08)
            shift = 600.0 * (.62, .78, .08)[k]
            c.eye[k] -= shift
            c.screen_origin[k] -= shift
        w, h = 96, 64
    elif case == "inside_sphere":
        _lattice(s, 5, 5, 3, 1.8, .75)
        eye = (-3 + 1.8 * 2 + .1, -1 + 1.8 * 2 - .2, .8 + 1.8)       # inside the sphere (2, 2, 1)
        for k in range(3):
            delta = eye[k] - c.eye[k]
            c.eye[k] += delta
            c.screen_origin[k] += delta
    elif case == "jittered":
        _lattice(s, 7, 7, 3, 1.5, .5, jitter=.5, rvar=.8, seed=7)
    elif case == "row_of_200":
        for i in range(200):
            s.addSphere((-40 + 1.0 * i, 6 + .01 * i, .45), .4).setColor(i % 2, .5, 1 - i % 2).setReflectiveFactor(.7 if i % 3 == 0 else 0.0)
    elif case == "dense_small":
        _lattice(s, 12, 12, 3, .5, .2, jitter=.05, rvar=.2, seed=3)
    else:
        s.addSphere((3, -5, 9), .2).setAsLightSource(.6)
        _lattice(s, 6, 6, 2, 1.8, .75)
    p = api.default_params(w, h, d)
    gpu_ctx.upload_flat(s.flatten(), c)
    assert gpu_ctx.scene_structures()["grid_cells"] > 0, gpu_ctx.scene_structures()      # the scene does take the grid kernel
    img, stats = gpu_ctx.render(p)
    want, cnt = O.render(s.flatten(), c, p)
    assert_bit_identical(img, want, f"sphere grid: {case}")
    check_counters(stats, cnt)


@pytest.mark.parametrize("spec,w,h,d", [("lattice:1:4", 160, 128, 12), ("lattice:2:5", 128, 96, 8), ("lattice:3:3", 96, 80, 30),
                                        ("lattice:4:6", 128, 96, 6), ("lattice:7:8", 96, 64, 10)])
def test_named_lattice_scenes_take_the_grid_and_match_the_oracle(gpu_ctx, spec, w, h, d):
    """The jittered lattices of scenes/scene_builders.inc (the oracle is pinned to the reference binary on the same
    scenes, tests/test_oracle.py): touching and overlapping spheres, two or three lights, mirrors and diffuse-0 spheres."""
    scene, cam = make_scene(spec)
    p = api.default_params(w, h, d)
    gpu_ctx.upload(scene, cam)
    assert gpu_ctx.scene_structures()["grid_cells"] > 0
    img, stats = gpu_ctx.render(p)
    want, cnt = O.render(scene.flatten(), cam.export(), p)
    assert_bit_identical(img, want, spec)
    check_counters(stats, cnt)


@pytest.mark.gpu
@pytest.mark.parametrize("name,w,h,d", [("synth256", 1920, 1080, 10), ("default", 3840, 2160, 50), ("default", 1920, 1080, 5)])
def test_chunked_host_render_equals_single_launch(gpu_ctx, name, w, h, d):
    """A band that goes to host memory is rendered as column chunks, their launches round robin on several streams
    with the copies behind them (render_submit); a band that stays on the device is one launch.  Same frame, same
    ray counters — into pinned and into pageable memory, and with two such frames in flight."""
    scene, cam = make_scene(name)
    p = api.default_params(w, h, d)
    gpu_ctx.upload(scene, cam)
    st_dev = gpu_ctx.render_device(p)
    want = gpu_ctx.download(np.empty((w, h, 3), np.float32)).copy()
    assert st_dev.gpu_launches == 1
    hb = [api.HostBuffer(w * h * 12) for _ in range(2)]
    outs = [b.array(np.float32, (w, h, 3)) for b in hb]
    outs[0][:] = -1.0
    img, st = gpu_ctx.render(p, out=outs[0])
    assert st.gpu_launches > 1, "expected a chunked render"
    assert np.array_equal(bits(img), bits(want)) and st.rays == st_dev.rays
    img2, st2 = gpu_ctx.render(p)          # pageable numpy memory
    assert np.array_equal(bits(img2), bits(want)) and st2.rays == st_dev.rays
    for o in outs:
        o[:] = -1.0
    tickets = [gpu_ctx.render_async(p, out=o) for o in outs]
    for t, o in zip(tickets, outs):
        assert gpu_ctx.wait(t).rays == st_dev.rays
        assert np.array_equal(bits(o), bits(want))
