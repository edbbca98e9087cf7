"""CPU tests: the host construction API (include/CelioRayTracer.hpp, tcrt_host.h) and the
C-ABI surface of libtcrt.so.  No compute calls: there is no GPU here and no CPU fallback."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from oracle import oracle_py as O
from tilecoderaytracer_b200 import _ffi, api

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32


def arr(ptr, n):
    return np.ctypeslib.as_array(ptr, shape=(n,)).copy()


# ---- ABI surface -----------------------------------------------------------------------------

def declared_symbols():
    names = set()
    for h in ("tcrt.h", "tcrt_host.h"):
        src = open(os.path.join(ROOT, "include", h)).read()
        src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
        names |= set(re.findall(r"\b(tcrt_\w+)\s*\(", src))
    return names


def test_library_exports_every_declared_symbol():
    lib = _ffi.load()
    decl = declared_symbols()
    assert len(decl) >= 40
    for name in sorted(decl):
        assert hasattr(lib, name), f"{name} declared in include/*.h but not exported by libtcrt.so"
    # and the Python binding table covers exactly the declared set
    assert set(_ffi.SIGNATURES) == decl
    out = subprocess.run(["nm", "-D", "--defined-only", _ffi.LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r" T (tcrt_\w+)", out))
    assert decl <= exported


def test_library_is_sm100a_only_and_has_no_oracle_dependency():
    out = subprocess.run(["cuobjdump", "-lelf", _ffi.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert not re.search(r"sm_(?!100a)\d+", out), out
    ldd = subprocess.run(["ldd", _ffi.LIB_PATH], capture_output=True, text=True).stdout
    assert "liboracle" not in ldd
    strings = subprocess.run(["strings", _ffi.LIB_PATH], capture_output=True, text=True).stdout
    assert "tcrt_oracle_render" not in strings


NO_DEVICE_CHECK = """
import ctypes as C, sys
sys.path.insert(0, %r)
from tilecoderaytracer_b200 import _ffi, api
lib = _ffi.load()
n = lib.tcrt_device_count()
assert n in (_ffi.TCRT_ERR_NO_DEVICE, 0), n
h = C.c_void_p()
rc = lib.tcrt_create(C.byref(h), None, 1)
assert rc == _ffi.TCRT_ERR_NO_DEVICE and not h.value, rc
assert b"CUDA" in lib.tcrt_last_error(None) or b"device" in lib.tcrt_last_error(None)
try:
    api.Context([0])
except api.TcrtError:
    print("NO_DEVICE_OK")
""" % ROOT


def test_no_gpu_means_loud_failure_not_fallback():
    """In a process that sees no CUDA device (CUDA_VISIBLE_DEVICES empty, so that this runs on a GPU machine too)."""
    r = subprocess.run([sys.executable, "-c", NO_DEVICE_CHECK], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True)
    assert r.returncode == 0 and "NO_DEVICE_OK" in r.stdout, r.stdout + r.stderr


def test_abi_version_and_default_params():
    lib = _ffi.load()
    assert lib.tcrt_abi_version() == 2
    p = api.default_params()
    # rt_project_parameters.h:65-66,73-74, RayTracer.h:52
    assert (p.width, p.height, p.max_depth, p.shadows_on, p.reflections_on) == (500, 504, 50, 1, 1)
    assert list(p.null_color) == [0.75, 0.75, 0.75] and p.far_dist == 65535.0


def test_txt_header_matches_reference_file(golden):
    """init_log + the three tags of printPixelsToLog, against the as-is program's own file."""
    want = golden["asis"]["rt_asis"]["header_lines"]
    rt = float(want[7].split(":")[1].rstrip("."))
    got = api.txt_header(api.default_params(), rt).decode().splitlines()
    assert got[:7] == want[:7]
    assert got[7] == want[7]                       # Run_Time:%f.
    assert got[8].startswith("us/pixel:") and got[9] == want[9]
    assert abs(float(got[8].split(":")[1].rstrip(".")) - rt * 1e6 / (500 * 504)) < 1e-5
    big = api.txt_header(api.default_params(7680, 4320, 10), 0.0).decode().splitlines()
    assert big[1] == "Horizontal_Resolution:7680." and big[2] == "Vertical_Resolution:4320."


# ---- camera ------------------------------------------------------------------------------------

def test_camera_default_pose_and_eye_rays():
    cam = api.Camera()
    c = cam.export()
    # Camera.cpp:22-38: horizontal ∝ (.1,-.08,0), vertical = horizontal x outward, eye one unit behind
    h = np.array(c.horizontal[:], f32)
    v = np.array(c.vertical[:], f32)
    hx = f32(.1) / np.sqrt(f32(.1) * f32(.1) + f32(-.08) * f32(-.08) + f32(0), dtype=f32)
    assert h[0] == f32(hx) and h[2] == 0
    assert abs(float(np.dot(h, v))) < 1e-6 and abs(float(np.linalg.norm(v)) - 1) < 1e-6
    assert list(c.screen_origin) == [-4.0, -4.0, 1.5]
    assert (c.screen_width, c.screen_height, c.screen_halfwidth, c.screen_halfheight) == (1, 1, .5, .5)
    eye = np.array(c.eye[:], f32)
    assert abs(float(np.linalg.norm(eye - np.array([-4, -4, 1.5], f32))) - 1) < 1e-6
    # createEyeRay (host) == primary-ray generation of the oracle, bit for bit
    p = api.default_params(37, 23, 5)
    for x, z in [(0, 0), (36, 22), (17, 5), (1, 21)]:
        o1, d1 = cam.createEyeRay(f32(x) / f32(37), f32(z) / f32(23))
        o2, d2 = O.primary_ray(c, p, x, z)
        assert np.array_equal(o1.view(np.uint32), o2.view(np.uint32))
        assert np.array_equal(d1.view(np.uint32), d2.view(np.uint32))
        assert abs(float(np.linalg.norm(d1)) - 1) < 1e-6


def test_camera_two_mirrors_pose():
    cam = api.Camera()
    cam.setSceneTwoMirrors()
    c = cam.export()
    assert list(c.screen_origin) == [0, 0, 2.5]
    assert list(c.horizontal) == [1, 0, 0] and list(c.vertical) == [0, 0, 1]
    assert list(c.eye) == [0, -1, 2.5]


# ---- scenes ---------------------------------------------------------------------------------------

def test_default_scene_object_list():
    """SURVEY appendix A / Scene.cpp:209-387."""
    s = api.Scene().initialize()
    assert s.getObjectCount() == 32
    f = s.flatten()
    assert (f.n_spheres, f.n_inf_planes, f.n_fin_planes, f.n_lights, f.n_textures) == (7, 1, 24, 2, 1)
    assert arr(f.sphere_obj, 7).tolist() == [0, 1, 2, 3, 4, 5, 6]
    assert arr(f.inf_obj, 1).tolist() == [7]
    assert arr(f.fin_obj, 24).tolist() == list(range(8, 32))
    assert arr(f.light_obj, 2).tolist() == [0, 1]
    sg = arr(f.sphere_geom, 28).reshape(7, 4)
    assert sg[0].tolist() == [f32(6.99), f32(6.99), 5.5, f32(f32(.15) * f32(.15))]
    assert sg[2].tolist() == [0, 0, 2, 1] and sg[5].tolist() == [0, 3, 1, 1] and sg[4][0] == -2.5
    surf = arr(f.obj_surface, 128).reshape(32, 4)
    mat = arr(f.obj_material, 128).reshape(32, 4)
    info = arr(f.obj_info, 128).reshape(32, 4)
    assert mat[0][2] == 0.75 and mat[1][2] == 1.0 and info[0][2] == 1 and info[2][2] == 0
    assert surf[2].tolist() == [1, 0, 0, 1] and mat[2][1] == 1.0          # red mirror ball
    assert surf[5].tolist() == [1, 1, 1, 0] and mat[5][1] == 1.0          # pure mirror, diffuse 0
    assert mat[4][0] == 0.5                                               # specular .5
    assert surf[7].tolist() == [0, 1, 0, 0.5] and mat[7][1] == 0.5 and info[7][3] == 0   # checker ground
    assert arr(f.textures, 8).tolist() == [1, 1, 1, 3, 0, 0, 0, 3]
    assert surf[8].tolist() == [f32(.2), f32(.2), 0, 1]                   # pedestal
    assert mat[14][0] == f32(.2) and surf[20][0] == f32(.33) and mat[20][0] == 0
    assert surf[26][0] == f32(2 / 3.) and mat[26][1] == 0.5 and mat[26][0] == 0.5


def test_make_scene_box_faces():
    """Scene.cpp:392-416: corners and the (origin, vertical corner, horizontal corner) face order."""
    s = api.Scene()
    faces = s.makeSceneBox((-7, -7, -1), (14, 14, 7))
    assert [o.index for o in faces] == list(range(6))
    f = s.flatten()
    g = arr(f.fin_geom, 6 * 16).reshape(6, 4, 4)
    org = arr(f.obj_origin, 24).reshape(6, 4)
    # face 0 = (c0, c3, c2): origin c0, vertical along +z (7), horizontal along +y (14)
    assert g[0][3][:3].tolist() == [-7, -7, -1]
    assert g[0][1].tolist() == [0, 1, 0, 14] and g[0][2].tolist() == [0, 0, 1, 7]
    assert g[0][0][:3].tolist() == [1, 0, 0]            # normal = horizontal x vertical
    assert g[0][0][3] == -7.0                           # -distance_to_origin = origin . normal
    # SceneObject origin moves to the far corner (SceneFinitePlane.cpp:74-79)
    assert org[0][:3].tolist() == [-7, 7, 6]
    # face 3 = (c7, c4, c6): origin c7
    assert g[3][3][:3].tolist() == [7, 7, 6]
    nrm = arr(f.obj_normals, 48).reshape(6, 2, 4)
    assert np.allclose(nrm[:, 0, :3], -nrm[:, 1, :3])


def test_finite_plane_axes_ctor_and_infinite_plane():
    s = api.Scene()
    s.addFinitePlaneAxes((-1.75, 7, 0), (0, -1, 0), (1, 0, 0), 5, 3.5)
    s.addInfinitePlane((0, 0, 0), (0, 0, 2), (3, 0, 0))
    f = s.flatten()
    g = arr(f.fin_geom, 16).reshape(4, 4)
    assert g[0].tolist() == [0, -1, 0, -7]       # normal, -dto = o.n = -7
    assert g[1].tolist() == [1, 0, 0, 3.5] and g[2][3] == 5
    assert g[2][:3].tolist() == [0, 0, 1]        # vertical = normal x horizontal
    ig = arr(f.inf_geom, 16).reshape(4, 4)
    assert ig[0].tolist() == [0, 0, 1, 0] and ig[1][:3].tolist() == [1, 0, 0] and ig[2][:3].tolist() == [0, 1, 0]
    nrm = arr(f.obj_normals, 16).reshape(2, 2, 4)
    assert nrm[1][1][:3].tolist() == [0, 0, -1]
    # the reference negates with 0 - c (vector3d.h:113): the zero components stay +0
    assert not np.signbit(nrm[1][1][0]) and not np.signbit(nrm[1][1][1])


def test_material_defaults_and_setters():
    s = api.Scene()
    o = s.addSphere((1, 2, 3), 2.0)
    f = s.flatten()
    # ObjMaterial.h:13-21; SceneObject(origin) ctor leaves diffuse at 1
    assert arr(f.obj_surface, 4).tolist() == [1, 1, 1, 1] and arr(f.obj_material, 4).tolist() == [1, 0, 1, 0]
    o.setColor(.25, .5, .75).setDiffuseFactor(.1).setSpecularFactor(.2).setReflectiveFactor(.3)
    o.setAsLightSource(.6)
    o.setCheckerBoard((1, 0, 0), (0, 0, 1), 2.5, 1.5)
    f = s.flatten()
    assert arr(f.obj_surface, 4).tolist() == [.25, .5, .75, f32(.1)]
    assert arr(f.obj_material, 4).tolist() == [f32(.2), f32(.3), f32(.6), 0]
    assert arr(f.obj_info, 4).tolist() == [0, 0, 1, 0] and f.n_lights == 1 and f.n_textures == 1
    assert arr(f.textures, 8).tolist() == [1, 0, 0, 2.5, 0, 0, 1, 1.5]
    assert arr(f.sphere_geom, 4).tolist() == [1, 2, 3, 4]


def test_add_object_refuses_at_capacity(capfd):
    """Scene::addObject: `object_count+1 >= MAX_OBJECT_COUNT` -> message, no add (Scene.cpp:470-479)."""
    s = api.Scene()
    for i in range(3999):
        s.addSphere((i, 0, 0), 1)
    assert s.getObjectCount() == 3999
    with pytest.raises(api.TcrtError):
        s.addSphere((0, 0, 0), 1)
    assert s.getObjectCount() == 3999
    assert "Added too many objects" in capfd.readouterr().out


def test_two_mirrors_and_synthetic_counts():
    cam = api.Camera()
    s = api.Scene().initializeTwoMirrors(cam)
    assert s.getObjectCount() == 3920            # Scene.cpp:131 "3920 we need this number of objects"
    f = s.flatten()
    assert (f.n_spheres, f.n_inf_planes, f.n_fin_planes, f.n_lights) == (3915, 1, 4, 1)
    assert list(cam.export().eye) == [0, -1, 2.5]
    assert api.Scene().build("synth1024").getObjectCount() == 1027
    assert api.Scene().build("synth256").getObjectCount() == 259
    with pytest.raises(api.TcrtError):
        api.Scene().build("no_such_scene")


def test_finite_plane_threshold_is_a_float_compare():
    """`t < 1E-5` is a double compare in the reference (SceneFinitePlane.cpp:102); the kernels
    use t <= 9.99999974738e-06f.  Equivalent for every float around the threshold."""
    thr = f32(9.99999974738e-06)
    assert float(thr) < 1e-5 < float(np.nextafter(thr, f32(1)))
    t = thr
    for _ in range(2000):
        t = np.nextafter(t, f32(0))
    for _ in range(4000):
        assert (float(t) < 1e-5) == bool(t <= thr)
        t = np.nextafter(t, f32(1))
    for special in (f32(0), f32(-0.0), f32(-1), f32(np.inf), f32(np.nan)):
        assert (float(special) < 1e-5) == bool(special <= thr)


def test_partition_tiles_the_image():
    from tilecoderaytracer_b200.partition import column_band, column_bands

    for w in (1, 7, 500, 1920, 3840, 7680):
        for n in (1, 2, 3, 4, 8):
            bands = column_bands(w, n)
            assert bands[0][0] == 0 and bands[-1][1] == w
            assert all(a[1] == b[0] for a, b in zip(bands, bands[1:]))
            assert max(b - a for a, b in bands) - min(b - a for a, b in bands) <= 1
    with pytest.raises(ValueError):
        column_band(10, 2, 2)


def test_cost_balanced_bands_tile_and_balance():
    """tcrt_bands_from_costs (host only): bands tile [0, W), are monotone, and equalise the cost."""
    from tilecoderaytracer_b200.partition import bands_from_costs, column_bands

    rng = np.random.default_rng(7)
    for w, n, groups in [(1920, 8, 256), (7680, 8, 256), (500, 3, 250), (64, 8, 64), (5, 8, 5), (1000, 1, 10)]:
        costs = rng.random(groups) * 10 + (np.arange(groups) > groups // 2) * 30     # right half 4x as expensive
        bands = bands_from_costs(costs, w, n)
        assert bands[0][0] == 0 and bands[-1][1] == w
        assert all(a[1] == b[0] for a, b in zip(bands, bands[1:])) and all(x0 <= x1 for x0, x1 in bands)
        if w >= 500 and n > 1:
            per_col = np.repeat(costs, int(np.ceil(w / groups)))[:w] if w % groups else np.repeat(costs, w // groups)
            load = [per_col[x0:x1].sum() for x0, x1 in bands]
            assert max(load) <= 1.15 * (sum(load) / n)
            eq = [per_col[x0:x1].sum() for x0, x1 in column_bands(w, n)]
            assert max(load) < max(eq)
    # uniform and all-zero costs give the equal-width cut
    assert bands_from_costs([1.0] * 64, 640, 4) == column_bands(640, 4)
    assert bands_from_costs([0.0] * 10, 640, 4) == column_bands(640, 4)
    with pytest.raises(ValueError):
        bands_from_costs([1.0, -1.0], 10, 2)


def test_rebalance_feedback_converges():
    """tcrt_rebalance_columns (host only): iterating on a synthetic cost profile equalises band times."""
    from tilecoderaytracer_b200.partition import column_bands, rebalance

    w, n = 1920, 8
    x = np.arange(w)
    density = 1.0 + 4.0 * np.exp(-((x - 800) / 150.0) ** 2) + 2.0 * (x > 1500)      # a hot spot and a plateau
    bands = column_bands(w, n)
    for _ in range(4):
        ms = [density[x0:x1].sum() for x0, x1 in bands]
        bands = rebalance(bands, ms, w)
        assert bands[0][0] == 0 and bands[-1][1] == w and all(a[1] == b[0] for a, b in zip(bands, bands[1:]))
    ms = [density[x0:x1].sum() for x0, x1 in bands]
    assert max(ms) <= 1.03 * (sum(ms) / n)
    with pytest.raises(ValueError):
        rebalance([(0, 5), (5, 9)], [1.0, 1.0], 10)


def test_text_scene_loader_reproduces_the_default_scene(tmp_path):
    """scenes/default.scene through tcrt_hscene_load_text flattens to exactly the arrays of
    Scene::initialize() (Scene.cpp:209-387); errors carry the line number."""
    import ctypes as C
    import os

    from tilecoderaytracer_b200 import _ffi

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sa = api.Scene().initialize()       # the flattened views point into storage owned by the scenes
    sb = api.Scene().load_text(os.path.join(root, "scenes", "default.scene"))
    a, b = sa.flatten(), sb.flatten()
    for name, ctype in _ffi.TcrtScene._fields_:
        va, vb = getattr(a, name), getattr(b, name)
        if isinstance(va, int):
            assert va == vb, name
    n = a.n_objects
    sizes = {"sphere_geom": 4 * a.n_spheres, "fin_geom": 16 * a.n_fin_planes, "inf_geom": 16 * a.n_inf_planes,
             "obj_surface": 4 * n, "obj_material": 4 * n, "obj_origin": 4 * n, "obj_normals": 8 * n,
             "textures": 8 * a.n_textures}
    for name, cnt in sizes.items():
        xa = np.ctypeslib.as_array(getattr(a, name), (cnt,)).view(np.uint32)
        xb = np.ctypeslib.as_array(getattr(b, name), (cnt,)).view(np.uint32)
        assert np.array_equal(xa, xb), name
    for name, cnt in {"obj_info": 4 * n, "sphere_obj": a.n_spheres, "fin_obj": a.n_fin_planes,
                      "inf_obj": a.n_inf_planes, "light_obj": a.n_lights}.items():
        assert np.array_equal(np.ctypeslib.as_array(getattr(a, name), (cnt,)),
                              np.ctypeslib.as_array(getattr(b, name), (cnt,))), name
    bad = tmp_path / "bad.scene"
    bad.write_text("sphere 0 0 0 1\ncolor 1 0\n")
    with pytest.raises(api.TcrtError, match="line 2"):
        api.Scene().load_text(str(bad))
    bad.write_text("color 1 0 0\n")
    with pytest.raises(api.TcrtError, match="before any primitive"):
        api.Scene().load_text(str(bad))
    with pytest.raises(api.TcrtError):
        api.Scene().load_text(str(tmp_path / "missing.scene"))


def test_txt_to_ppm_tool(tmp_path):
    """tools/txt_to_ppm.py (the offline viewer replacement): tags + pixel lines -> PPM rows, top first."""
    import importlib.util
    import os

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("txt_to_ppm", os.path.join(root, "tools", "txt_to_ppm.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    w, h = 3, 2
    px = np.zeros((w, h, 3))
    px[0, 0] = (1.0, 0.5, 0.0)       # bottom-left
    px[2, 1] = (2.5, 0.25, 0.999)    # top-right, over-range red
    p = api.default_params(w, h, 5)
    txt = api.txt_header(p, 0.0) + b"".join(b"(%f, %f, %f)\n" % tuple(px[x, z]) for x in range(w) for z in range(h))
    path = tmp_path / "s.txt"
    path.write_bytes(txt)
    gw, gh, got, tags = mod.read_txt(str(path))
    assert (gw, gh) == (w, h) and np.allclose(got, px) and tags["Hardware_Target"] == "OSX C++"
    img = mod.to_image(mod.quant8(got))
    assert img.shape == (h, w, 3)
    assert tuple(img[1, 0]) == (255, 128, 0) and tuple(img[0, 2]) == (255, 64, 255)


def test_txt_create_sizes_the_file_for_fixed_width_lines(tmp_path):
    """tcrt_txt_create (host only): header + room for W*H pixel lines of 31 bytes, so that every rank of a
    one-process-per-GPU run can write its band at its place (tcrt_write_txt_band) without a gather."""
    p = api.default_params(40, 30, 5)
    path = str(tmp_path / "raytracer_screen.txt")
    api.txt_create(p, path, 1.5)
    head = api.txt_header(p, 1.5)
    data = open(path, "rb").read()
    assert data.startswith(head) and len(data) == len(head) + 40 * 30 * 31
    assert head.decode().splitlines()[7] == "Run_Time:1.500000."
    with pytest.raises(api.TcrtError) as e:
        api.txt_create(p, str(tmp_path / "no_such_dir" / "x.txt"), 0.0)
    assert e.value.code == _ffi.TCRT_ERR_IO


# ---- which pruning structures a scene gets (tcrt_plan_scene: the host half of tcrt_upload_scene, no device) ------------

def _plan(name):
    cam = api.Camera()
    scene = api.Scene().build(name, cam)       # owns the arrays flatten() points into
    return api.plan_scene(scene.flatten())


def test_plan_scene_of_the_baseline_scenes():
    """The structures behind the five BASELINE configs and the reference's SCENE 2: box clusters for the default scene's
    24 rectangles, BVH + uniform grid in step with the lattice for the synthetic scenes (one cell per lattice site plus
    the margin cells), BVH alone for SCENE 2 (its radius-10 sphere is 4x the median: no grid)."""
    d = _plan("default")
    assert (d["clusters"], d["cluster_rects"], d["bvh_spheres"], d["grid_cells"], d["linear_spheres"]) == (4, 24, 0, 0, 7)
    s = _plan("synth256")
    assert s["bvh_spheres"] == 256 and s["grid_dims"] == (9, 9, 5) and s["grid_cells"] == 405 and s["linear_spheres"] == 2
    s = _plan("synth1024")
    assert s["bvh_spheres"] == 1024 and s["grid_dims"] == (17, 17, 5) and s["linear_spheres"] == 2
    t = _plan("two_mirrors")
    assert t["bvh_spheres"] > 3900 and t["grid_cells"] == 0 and t["linear_finite"] == 4
    assert all(v["staged_bytes"] <= 200 * 1024 for v in (d, s, t))


_keep = []       # scenes own the arrays their flattened views point into


def _sphere_scene(centres, radius):
    s = api.Scene()
    _keep.append(s)
    s.addSphere((-2, -6, 12), .15).setAsLightSource(.75)
    s.addInfinitePlane((0, 0, 0), (0, 0, 1), (1, 0, 0))
    for c, r in zip(centres, radius):
        s.addSphere(tuple(float(x) for x in c), float(r))
    return s.flatten()


def test_plan_scene_grid_acceptance_rules():
    """tcrt_build_sphere_grid takes lattice-like sets only: at least 24 similar spheres; one sphere four times the median,
    or spheres so crowded that a cell would hold more than 24, and the BVH stays alone."""
    lattice = [(1.5 * i, 1.5 * j, .6 + 1.5 * k) for k in range(2) for j in range(4) for i in range(4)]      # 32 sites
    ok = api.plan_scene(_sphere_scene(lattice, [.5] * 32))
    assert ok["grid_cells"] > 0 and ok["bvh_spheres"] == 32 and min(ok["grid_dims"]) >= 2
    few = api.plan_scene(_sphere_scene(lattice[:20], [.5] * 20))
    assert few["grid_cells"] == 0
    giant = api.plan_scene(_sphere_scene(lattice + [(40, 40, 12)], [.5] * 32 + [11.0]))
    assert giant["grid_cells"] == 0 and giant["bvh_spheres"] == 33
    rng = np.random.default_rng(5)
    heap = [(3 + .02 * rng.random(), 3 + .02 * rng.random(), 1 + .02 * rng.random()) for _ in range(60)]     # 60 nearly coincident
    crowded = api.plan_scene(_sphere_scene(heap, [.5] * 60))
    assert crowded["grid_cells"] == 0
    jitter = [(x + .3 * rng.random(), y + .3 * rng.random(), z + .3 * rng.random()) for x, y, z in lattice]
    j = api.plan_scene(_sphere_scene(jitter, list(.4 + .2 * rng.random(32))))
    assert j["grid_cells"] > 0


def test_plan_scene_rejects_what_upload_rejects():
    flat = _sphere_scene([(0, 0, 1)], [.5])
    flat.n_spheres += 1                       # counts no longer add up
    with pytest.raises(api.TcrtError) as e:
        api.plan_scene(flat)
    assert e.value.code == _ffi.TCRT_ERR_INVALID


def _grid_soundness(flat, spheres, seed):
    """DESIGN.md 4.5 (i): a sphere the reference hits at distance d is met inside the sphere fattened by at most
    grid_margin, and that point must lie in a cell where the sphere is registered.  Checked for random points of every
    sphere's volume and of its shell out to the margin.  spheres: [(object index, centre, radius)]."""
    rng = np.random.default_rng(seed)
    _, margin = api.plan_grid_cells(flat, [(0, 0, 0)])
    assert margin > 0
    pts, owner = [], []
    for obj, c, r in spheres:
        u = rng.normal(size=(24, 3))
        u /= np.linalg.norm(u, axis=1, keepdims=True)
        rad = np.concatenate([r * rng.random(8) ** (1 / 3), np.full(8, r), r + margin * rng.random(8)])
        pts.append(np.asarray(c) + u * rad[:, None])
        owner += [obj] * 24
    cells, _ = api.plan_grid_cells(flat, np.concatenate(pts))
    missing = [(o, i) for i, (o, reg) in enumerate(zip(owner, cells)) if o not in reg]
    assert not missing, f"{len(missing)} of {len(owner)} points lie in a cell that does not list their sphere, e.g. {missing[:3]}"
    return max(len(reg) for reg in cells)


@pytest.mark.parametrize("name", ["synth256", "synth1024"])
def test_sphere_grid_registers_every_sphere_wherever_it_can_be_hit(name):
    cam = api.Camera()
    scene = api.Scene().build(name, cam)
    flat = scene.flatten()
    n = flat.n_spheres
    geom = np.ctypeslib.as_array(flat.sphere_geom, shape=(n, 4))
    objs = np.ctypeslib.as_array(flat.sphere_obj, shape=(n,))
    info = np.ctypeslib.as_array(flat.obj_info, shape=(flat.n_objects, 4))
    spheres = [(int(o), g[:3].copy(), float(np.sqrt(g[3]))) for g, o in zip(geom, objs) if info[o, 2] == 0]
    assert len(spheres) == api.plan_scene(flat)["bvh_spheres"]
    assert _grid_soundness(flat, spheres, 11) == 1          # in step with the lattice: one sphere per cell


@pytest.mark.parametrize("spec", ["lattice:1:4", "lattice:2:5", "lattice:3:3", "lattice:4:6", "lattice:7:8"])
def test_sphere_grid_soundness_on_named_lattice_scenes(spec):
    cam = api.Camera()
    scene = api.Scene().build(spec, cam)
    flat = scene.flatten()
    n = flat.n_spheres
    geom = np.ctypeslib.as_array(flat.sphere_geom, shape=(n, 4))
    objs = np.ctypeslib.as_array(flat.sphere_obj, shape=(n,))
    info = np.ctypeslib.as_array(flat.obj_info, shape=(flat.n_objects, 4))
    spheres = [(int(o), g[:3].copy(), float(np.sqrt(g[3]))) for g, o in zip(geom, objs) if info[o, 2] == 0]
    plan = api.plan_scene(flat)
    assert plan["grid_cells"] > 0 and plan["bvh_spheres"] == len(spheres)
    _grid_soundness(flat, spheres, 7)


def test_sphere_grid_soundness_on_jittered_lattices():
    for seed in (1, 2, 3):
        rng = np.random.default_rng(seed)
        centres = [(1.5 * i + .5 * rng.random(), 1.5 * j + .5 * rng.random(), .8 + 1.5 * k + .5 * rng.random())
                   for k in range(3) for j in range(5) for i in range(5)]
        radii = list(.35 + .3 * rng.random(len(centres)))
        flat = _sphere_scene(centres, radii)
        assert api.plan_scene(flat)["grid_cells"] > 0
        # objects: light 0, plane 1, spheres from 2 (see _sphere_scene)
        spheres = [(2 + i, np.array(c), r) for i, (c, r) in enumerate(zip(centres, radii))]
        assert _grid_soundness(flat, spheres, 100 + seed) >= 2      # spheres straddle cells here


def test_sphere_grid_soundness_fuzz():
    """Anisotropic spacings, radius ratios up to 3.5, strong jitter, clumps: whatever tcrt_build_sphere_grid decides, a grid
    it builds registers every sphere wherever it can be hit (and a set it refuses simply keeps the BVH)."""
    rng = np.random.default_rng(2026)
    built = 0
    for trial in range(40):
        nx, ny, nz = (int(v) for v in rng.integers(2, 7, size=3))
        sp = rng.uniform(.6, 2.5, size=3)
        r0 = float(rng.uniform(.15, .6) * sp.min())
        ratio = float(rng.uniform(1.0, 3.5))
        jitter = float(rng.uniform(0.0, .6))
        centres, radii = [], []
        for k in range(nz):
            for j in range(ny):
                for i in range(nx):
                    c = np.array([i, j, k]) * sp + jitter * sp * (rng.random(3) - .5) + np.array([-3, -1, 3.0])
                    centres.append(tuple(float(v) for v in c))
                    radii.append(r0 * float(rng.uniform(1.0, ratio)))
        if trial % 5 == 0:                       # a clump of near-coincident spheres inside the lattice
            for _ in range(int(rng.integers(3, 12))):
                centres.append(tuple(float(v) for v in np.array(centres[0]) + .05 * rng.random(3)))
                radii.append(r0)
        flat = _sphere_scene(centres, radii)
        plan = api.plan_scene(flat)
        assert plan["bvh_spheres"] + plan["linear_spheres"] == len(centres) + 1          # + the light
        if plan["grid_cells"] == 0:
            continue
        built += 1
        assert max(plan["grid_dims"]) <= 64
        spheres = [(2 + i, np.array(c), r) for i, (c, r) in enumerate(zip(centres, radii))]
        in_grid = spheres if plan["bvh_spheres"] == len(spheres) else None
        if in_grid is not None:                  # every sphere is BVH- and therefore grid-covered
            _grid_soundness(flat, in_grid, 1000 + trial)
    assert built >= 10, f"only {built} of 40 sets got a grid: the fuzz no longer exercises the builder"
