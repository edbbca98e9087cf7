"""Thin Python face of libtcrt.so, for tests and bench.py.

Names follow the reference's domain (Scene, Camera, SceneSphere ... — SURVEY.md §8b); every
method forwards to the C ABI.  Nothing here computes pixels.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Optional, Sequence

import numpy as np

from . import _ffi
from ._ffi import TcrtCamera, TcrtParams, TcrtScene, TcrtStats


class TcrtError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"tcrt error {code}: {msg}")
        self.code = code


def _f3(v: Sequence[float]):
    return (C.c_float * 3)(float(v[0]), float(v[1]), float(v[2]))


class Camera:
    """CelioRayTracer::Camera (Camera.h:11-41): fixed default pose, setSceneTwoMirrors()."""

    def __init__(self):
        self._lib = _ffi.load()
        self._h = self._lib.tcrt_hcamera_new()

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.tcrt_hcamera_free(self._h)
            self._h = None

    def setSceneTwoMirrors(self) -> None:
        self._lib.tcrt_hcamera_set_two_mirrors(self._h)

    def aim(self, screen_origin: Sequence[float], horizontal: Sequence[float], outwards: Sequence[float]) -> "Camera":
        """Camera::aim, the reference's pose arithmetic (Camera.cpp:22-38): the screen's centre at screen_origin, its
        x axis along horizontal, the view along outwards, vertical = horizontal x outwards (before either is
        normalised), then all three normalised and the eye one unit behind the screen.  The screen size is kept; for
        another field of view edit screen_width / screen_height of export() with halfwidth = width / 2 and halfheight =
        height / 2, as the reference sets them.  Returns self."""
        self._lib.tcrt_hcamera_aim(self._h, _f3(screen_origin), _f3(horizontal), _f3(outwards))
        return self

    def createEyeRay(self, dx_percent: float, dy_percent: float):
        o = (C.c_float * 3)()
        d = (C.c_float * 3)()
        self._lib.tcrt_hcamera_eye_ray(self._h, dx_percent, dy_percent, o, d)
        return np.array(o[:], dtype=np.float32), np.array(d[:], dtype=np.float32)

    def export(self) -> TcrtCamera:
        cam = TcrtCamera()
        self._lib.tcrt_hcamera_export(self._h, C.byref(cam))
        return cam


def _camera_table(cameras) -> C.Array:
    """A contiguous tcrt_camera array of Camera objects and / or TcrtCamera structs."""
    cams = [c.export() if isinstance(c, Camera) else c for c in cameras]
    for c in cams:
        assert isinstance(c, TcrtCamera), "cameras: Camera or TcrtCamera"
    return (TcrtCamera * len(cams))(*cams)


class SceneObjectRef:
    """Handle to one object of a Scene: the SceneObject / ObjMaterial setters."""

    def __init__(self, scene: "Scene", index: int):
        self.scene = scene
        self.index = index

    def _ck(self, rc):
        if rc != 0:
            raise TcrtError(rc, "bad object handle")
        return self

    def setColor(self, r, g, b):
        return self._ck(self.scene._lib.tcrt_hobj_set_color(self.scene._h, self.index, r, g, b))

    def setDiffuseFactor(self, f):
        return self._ck(self.scene._lib.tcrt_hobj_set_diffuse(self.scene._h, self.index, f))

    def setSpecularFactor(self, f):
        return self._ck(self.scene._lib.tcrt_hobj_set_specular(self.scene._h, self.index, f))

    def setReflectiveFactor(self, f):
        return self._ck(self.scene._lib.tcrt_hobj_set_reflective(self.scene._h, self.index, f))

    def setAsLightSource(self, intensity: float = 1.0):
        return self._ck(self.scene._lib.tcrt_hobj_set_light(self.scene._h, self.index, intensity))

    def setCheckerBoard(self, light=(1, 1, 1), dark=(0, 0, 0), width=2.0, height=2.0):
        return self._ck(self.scene._lib.tcrt_hobj_set_checker(self.scene._h, self.index, _f3(light), _f3(dark),
                                                             width, height))


class Scene:
    """CelioRayTracer::Scene (Scene.h:15-44) + flatten()."""

    def __init__(self):
        self._lib = _ffi.load()
        self._h = self._lib.tcrt_hscene_new()

    def __del__(self):
        if getattr(self, "_h", None):
            self._lib.tcrt_hscene_free(self._h)
            self._h = None

    # named scenes ---------------------------------------------------------------------
    def build(self, name: str, camera: Optional[Camera] = None) -> "Scene":
        rc = self._lib.tcrt_hscene_build(self._h, camera._h if camera else None, name.encode())
        if rc != 0:
            raise TcrtError(rc, f"cannot build scene {name!r}")
        return self

    def load_text(self, path: str, camera: Optional[Camera] = None) -> "Scene":
        """Text scene description (format: include/tcrt_host.h, example: scenes/default.scene)."""
        err = C.create_string_buffer(256)
        rc = self._lib.tcrt_hscene_load_text(self._h, camera._h if camera else None, path.encode(), err, 256)
        if rc != 0:
            raise TcrtError(rc, f"{path}: {err.value.decode()}")
        return self

    def initialize(self) -> "Scene":
        return self.build("default")

    def initializeTwoMirrors(self, camera: Camera) -> "Scene":
        return self.build("two_mirrors", camera)

    # primitives -------------------------------------------------------------------------
    def _obj(self, idx: int) -> SceneObjectRef:
        if idx < 0:
            raise TcrtError(idx, "Added too many objects to scene")
        return SceneObjectRef(self, idx)

    def addSphere(self, origin, radius) -> SceneObjectRef:
        return self._obj(self._lib.tcrt_hscene_add_sphere(self._h, _f3(origin), radius))

    def addInfinitePlane(self, origin, normal, horizontal) -> SceneObjectRef:
        return self._obj(self._lib.tcrt_hscene_add_infinite_plane(self._h, _f3(origin), _f3(normal), _f3(horizontal)))

    def addFinitePlaneCorners(self, origin, vertical_corner, horizontal_corner) -> SceneObjectRef:
        return self._obj(self._lib.tcrt_hscene_add_finite_plane_corners(self._h, _f3(origin), _f3(vertical_corner),
                                                                        _f3(horizontal_corner)))

    def addFinitePlaneAxes(self, origin, normal, horizontal, v_dist, h_dist) -> SceneObjectRef:
        return self._obj(self._lib.tcrt_hscene_add_finite_plane_axes(self._h, _f3(origin), _f3(normal),
                                                                     _f3(horizontal), v_dist, h_dist))

    def makeSceneBox(self, origin, dims) -> list[SceneObjectRef]:
        first = self._lib.tcrt_hscene_add_box(self._h, _f3(origin), _f3(dims))
        if first < 0:
            raise TcrtError(first, "Added too many objects to scene")
        return [SceneObjectRef(self, first + k) for k in range(6)]

    def getObjectCount(self) -> int:
        return self._lib.tcrt_hscene_object_count(self._h)

    def flatten(self) -> TcrtScene:
        s = TcrtScene()
        rc = self._lib.tcrt_hscene_flatten(self._h, C.byref(s))
        if rc != 0:
            raise TcrtError(rc, "flatten failed")
        return s


def default_params(width=500, height=504, max_depth=50, shadows=True, reflections=True) -> TcrtParams:
    p = TcrtParams()
    _ffi.load().tcrt_default_params(C.byref(p))
    p.width, p.height, p.max_depth = int(width), int(height), int(max_depth)
    p.shadows_on, p.reflections_on = int(bool(shadows)), int(bool(reflections))
    return p


@dataclass
class RenderStats:
    n_devices: int = 0
    bands: list = field(default_factory=list)
    render_ms: list = field(default_factory=list)
    d2h_ms: list = field(default_factory=list)
    rays_primary: int = 0
    rays_shadow: int = 0
    rays_reflect: int = 0
    rays_per_device: list = field(default_factory=list)
    gpu_launches: int = 0

    @property
    def rays(self) -> int:
        return self.rays_primary + self.rays_shadow + self.rays_reflect

    @staticmethod
    def from_c(st: TcrtStats) -> "RenderStats":
        n = st.n_devices
        per_dev = [int(st.rays_primary[i] + st.rays_shadow[i] + st.rays_reflect[i]) for i in range(n)]
        return RenderStats(
            n_devices=n,
            bands=[(st.col_begin[i], st.col_end[i]) for i in range(n)],
            render_ms=[st.render_ms[i] for i in range(n)],
            d2h_ms=[st.d2h_ms[i] for i in range(n)],
            rays_primary=sum(int(st.rays_primary[i]) for i in range(n)),
            rays_shadow=sum(int(st.rays_shadow[i]) for i in range(n)),
            rays_reflect=sum(int(st.rays_reflect[i]) for i in range(n)),
            rays_per_device=per_dev,
            gpu_launches=int(st.gpu_launches),
        )


STRUCTURE_KEYS = ("bvh_spheres", "grid_cells", "bvh_finite", "clusters", "cluster_rects", "linear_spheres", "linear_finite",
                  "staged_bytes")


def plan_scene(flat) -> dict:
    """The pruning structures tcrt_upload_scene would build for a flattened scene (tcrt_plan_scene: host work only,
    no device); "grid_dims" = cells per axis of the sphere grid, (0, 0, 0) without one."""
    lib = _ffi.load()
    info, dims = (C.c_int * 8)(), (C.c_int * 3)()
    rc = lib.tcrt_plan_scene(C.byref(flat), info, dims)
    if rc != 0:
        raise TcrtError(rc, (lib.tcrt_last_error(None) or b"").decode())
    out = dict(zip(STRUCTURE_KEYS, (int(v) for v in info)))
    out["grid_dims"] = tuple(int(v) for v in dims)
    return out


def plan_grid_cells(flat, points, cap: int = 32):
    """For every row of points[n, 3]: the object indices registered in the grid cell that contains it (a list of sets),
    and the grid's margin — tcrt_plan_grid_cells, host only."""
    lib = _ffi.load()
    pts = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
    objs = np.full((len(pts), cap), -1, dtype=np.int32)
    counts = np.zeros(len(pts), dtype=np.int32)
    margin = C.c_float(0.0)
    rc = lib.tcrt_plan_grid_cells(C.byref(flat), pts.ctypes.data, len(pts), objs.ctypes.data, cap, counts.ctypes.data, C.byref(margin))
    if rc != 0:
        raise TcrtError(rc, (lib.tcrt_last_error(None) or b"").decode())
    assert counts.max(initial=0) <= cap, "raise cap"
    return [set(int(v) for v in objs[i, :counts[i]]) for i in range(len(pts))], float(margin.value)


def plan_dead_paths(flat, params: TcrtParams) -> bool:
    """Whether renders of the flattened scene with params may skip the shading of dead reflection levels
    (tcrt_plan_dead_paths, host only)."""
    lib = _ffi.load()
    prune = C.c_int(0)
    rc = lib.tcrt_plan_dead_paths(C.byref(flat), C.byref(params), C.byref(prune))
    if rc != 0:
        raise TcrtError(rc, (lib.tcrt_last_error(None) or b"").decode())
    return bool(prune.value)


def sphere_geom(centres, radii) -> np.ndarray:
    """The (n, 4) float32 rows Context.update_spheres takes: centre x y z, radius_squared, with radius_squared formed as
    SceneSphere(o, r) forms it — r * r in binary32."""
    c = np.asarray(centres, dtype=np.float32).reshape(-1, 3)
    r = np.asarray(radii, dtype=np.float32).reshape(-1)
    assert r.shape[0] == c.shape[0], "one radius per centre"
    out = np.empty((c.shape[0], 4), np.float32)
    out[:, :3] = c
    out[:, 3] = r * r
    return out


def material_rows(flat, objects):
    """The (surface, material, texture) rows of `objects` in a flattened scene, as Context.update_materials takes them:
    (n, 4) float32 (colour rgb, diffuse), (n, 4) float32 (specular, reflective, intensity, 0) and (n,) int32 texture ids.
    Edit a host Scene with the reference's setters, flatten it, and send the rows of the objects that changed."""
    idx = np.asarray(objects, dtype=np.int64).reshape(-1)
    n = flat.n_objects
    assert ((idx >= 0) & (idx < n)).all(), "object index out of range"
    if n == 0:
        return np.zeros((0, 4), np.float32), np.zeros((0, 4), np.float32), np.zeros(0, np.int32)
    surface = np.ctypeslib.as_array(flat.obj_surface, (n * 4,)).reshape(n, 4)
    material = np.ctypeslib.as_array(flat.obj_material, (n * 4,)).reshape(n, 4)
    info = np.ctypeslib.as_array(flat.obj_info, (n * 4,)).reshape(n, 4)
    return (np.ascontiguousarray(surface[idx], np.float32), np.ascontiguousarray(material[idx], np.float32),
            np.ascontiguousarray(info[idx, 3], np.int32))


def plane_rows(flat, objects):
    """The (geom, normals, origin) rows of the planes `objects` in a flattened scene, as Context.update_planes takes them:
    (n, 16) float32 in the layout of fin_geom or inf_geom by each object's type, (n, 8) float32 obj_normals rows (facing,
    then reverse normal) and (n, 4) float32 obj_origin rows.  Build the moved planes with the reference's constructors in a
    scene of the same object order, flatten it, and send the rows of the planes that moved."""
    idx = np.asarray(objects, dtype=np.int64).reshape(-1)
    n = flat.n_objects
    assert ((idx >= 0) & (idx < n)).all(), "object index out of range"
    geom = np.zeros((len(idx), 16), np.float32)
    if n == 0:
        return geom, np.zeros((0, 8), np.float32), np.zeros((0, 4), np.float32)
    info = np.ctypeslib.as_array(flat.obj_info, (n * 4,)).reshape(n, 4)
    tables = {}
    for kind, rows, count in ((1, "fin_geom", flat.n_fin_planes), (2, "inf_geom", flat.n_inf_planes)):
        if count:
            tables[kind] = np.ctypeslib.as_array(getattr(flat, rows), (count * 16,)).reshape(count, 16)
    for i, o in enumerate(idx):
        assert info[o, 0] in tables, f"object {o} is not a plane"
        geom[i] = tables[info[o, 0]][info[o, 1]]
    normals = np.ctypeslib.as_array(flat.obj_normals, (n * 8,)).reshape(n, 8)
    origin = np.ctypeslib.as_array(flat.obj_origin, (n * 4,)).reshape(n, 4)
    return (geom, np.ascontiguousarray(normals[idx], np.float32), np.ascontiguousarray(origin[idx], np.float32))


def normalize_like_reference(v) -> np.ndarray:
    """vector3d::normalize in numpy float32, as a Ray's constructor applies it: len = sqrtf((x*x + y*y) + z*z), then three
    IEEE divisions.  The ray-batch calls take directions as a Ray stores them; this turns raw directions (..., 3) into
    those, bit for bit."""
    a = np.asarray(v, dtype=np.float32)
    x, y, z = a[..., 0], a[..., 1], a[..., 2]
    with np.errstate(all="ignore"):
        length = np.sqrt((x * x + y * y) + z * z)
        return np.stack([x / length, y / length, z / length], axis=-1)


def _ray_inputs(origins, directions):
    """(n, origins, shared_origin, directions) as the ray-batch calls take them: float32, C-contiguous."""
    d = np.asarray(directions)
    assert d.dtype == np.float32 and d.ndim == 2 and d.shape[1] == 3 and d.flags["C_CONTIGUOUS"], "directions: (n, 3) float32"
    o = np.asarray(origins)
    assert o.dtype == np.float32 and o.flags["C_CONTIGUOUS"], "origins: float32, C-contiguous"
    shared = o.shape == (3,)
    assert shared or o.shape == d.shape, "origins: (n, 3), or (3,) for a shared origin"
    return d.shape[0], o, int(shared), d


class HostBuffer:
    """Pinned host memory (tcrt_alloc_host) viewed as a numpy array."""

    def __init__(self, nbytes: int):
        self._lib = _ffi.load()
        self.nbytes = int(nbytes)
        self.ptr = self._lib.tcrt_alloc_host(self.nbytes)
        if not self.ptr:
            raise TcrtError(_ffi.TCRT_ERR_CUDA, f"cannot pin {nbytes} bytes of host memory")

    def array(self, dtype, shape):
        buf = (C.c_char * self.nbytes).from_address(self.ptr)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def __del__(self):
        if getattr(self, "ptr", None):
            self._lib.tcrt_free_host(self.ptr)
            self.ptr = None


class Context:
    """tcrt_ctx: one or more B200s, a resident scene, the last rendered band."""

    def __init__(self, devices: Optional[Sequence[int]] = None):
        self._lib = _ffi.load()
        devs = list(devices) if devices is not None else [0]
        arr = (C.c_int * len(devs))(*devs)
        h = C.c_void_p()
        rc = self._lib.tcrt_create(C.byref(h), arr, len(devs))
        if rc != 0:
            raise TcrtError(rc, self._lib.tcrt_last_error(None).decode())
        self._h = h
        self.devices = devs

    def close(self):
        if getattr(self, "_h", None):
            self._lib.tcrt_destroy(self._h)
            self._h = None

    __del__ = close

    def _ck(self, rc: int):
        if rc != 0:
            raise TcrtError(rc, self._lib.tcrt_last_error(self._h).decode())

    def upload(self, scene: Scene, camera: Camera) -> None:
        flat = scene.flatten()
        cam = camera.export()
        self.upload_flat(flat, cam)

    def upload_flat(self, flat: TcrtScene, cam: TcrtCamera) -> None:
        self._ck(self._lib.tcrt_upload_scene(self._h, C.byref(flat), C.byref(cam)))
        self._n_lights = int(flat.n_lights)

    def scene_structures(self) -> dict:
        """Which pruning structures the uploaded scene got (tcrt_scene_structures)."""
        info = (C.c_int * 8)()
        self._ck(self._lib.tcrt_scene_structures(self._h, info))
        return dict(zip(STRUCTURE_KEYS, (int(v) for v in info)))

    def render(self, params: TcrtParams, x0: int = 0, x1: Optional[int] = None, out: Optional[np.ndarray] = None):
        """Render columns [x0,x1) to host memory; returns (array[x1-x0, H, 3] float32, RenderStats)."""
        x1 = params.width if x1 is None else x1
        shape = (x1 - x0, params.height, 3)
        if out is None:
            out = np.empty(shape, dtype=np.float32)
        assert out.dtype == np.float32 and out.size == int(np.prod(shape)) and out.flags["C_CONTIGUOUS"]
        st = TcrtStats()
        self._ck(self._lib.tcrt_render_columns(self._h, C.byref(params), x0, x1, out.ctypes.data_as(C.c_void_p),
                                               C.byref(st)))
        return out.reshape(shape), RenderStats.from_c(st)

    def render_device(self, params: TcrtParams, x0: int = 0, x1: Optional[int] = None) -> RenderStats:
        x1 = params.width if x1 is None else x1
        st = TcrtStats()
        self._ck(self._lib.tcrt_render_device(self._h, C.byref(params), x0, x1, C.byref(st)))
        return RenderStats.from_c(st)

    def render_async(self, params: TcrtParams, x0: int = 0, x1: Optional[int] = None, out: Optional[np.ndarray] = None) -> int:
        """Queue columns [x0,x1) of a frame (into `out`, pinned host memory, when given) and return a ticket at
        once; at most two frames are in flight.  wait(ticket) completes it."""
        x1 = params.width if x1 is None else x1
        if out is not None:
            assert out.dtype == np.float32 and out.size == (x1 - x0) * params.height * 3 and out.flags["C_CONTIGUOUS"]
        t = C.c_int(-1)
        self._ck(self._lib.tcrt_render_async(self._h, C.byref(params), x0, x1,
                                             out.ctypes.data_as(C.c_void_p) if out is not None else None, C.byref(t)))
        return t.value

    def render_rgb8(self, params: TcrtParams, x0: int = 0, x1: Optional[int] = None, out: Optional[np.ndarray] = None):
        """Columns [x0,x1) quantised to 8 bits on the GPU (q(c) = floor(clamp(c,0,1)*255 + 0.5)), 3 bytes per pixel to
        host memory; returns (array[x1-x0, H, 3] uint8, RenderStats).  x-major like render(): image rows (top row
        first) are a.transpose(1, 0, 2)[::-1].  The float frame stays on the device as the last render."""
        x1 = params.width if x1 is None else x1
        shape = (x1 - x0, params.height, 3)
        if out is None:
            out = np.empty(shape, dtype=np.uint8)
        assert out.dtype == np.uint8 and out.size == int(np.prod(shape)) and out.flags["C_CONTIGUOUS"]
        st = TcrtStats()
        self._ck(self._lib.tcrt_render_columns_rgb8(self._h, C.byref(params), x0, x1, out.ctypes.data_as(C.c_void_p),
                                                    C.byref(st)))
        return out.reshape(shape), RenderStats.from_c(st)

    def render_async_rgb8(self, params: TcrtParams, x0: int, x1: int, out: np.ndarray) -> int:
        """render_async() of an 8-bit frame into `out` (uint8, pinned host memory: HostBuffer.array(np.uint8, ...));
        wait(ticket) completes it."""
        assert out.dtype == np.uint8 and out.size == (x1 - x0) * params.height * 3 and out.flags["C_CONTIGUOUS"]
        t = C.c_int(-1)
        self._ck(self._lib.tcrt_render_async_rgb8(self._h, C.byref(params), x0, x1, out.ctypes.data_as(C.c_void_p),
                                                  C.byref(t)))
        return t.value

    def render_ss(self, params: TcrtParams, ss: int, x0: int = 0, x1: Optional[int] = None,
                  out: Optional[np.ndarray] = None):
        """Columns [x0,x1) of the supersampled frame: every pixel the mean of its ss x ss samples, sample (i, j) of pixel
        (x, z) being the reference's pixel (ss*x+i, ss*z+j) at (ss*W, ss*H), summed in the order of tcrt.h and resolved
        on the GPU.  Returns (array[x1-x0, H, 3] float32, RenderStats); the stats count the rays of the sample frame.
        The resolved frame becomes the last render."""
        x1 = params.width if x1 is None else x1
        shape = (x1 - x0, params.height, 3)
        if out is None:
            out = np.empty(shape, dtype=np.float32)
        assert out.dtype == np.float32 and out.size == int(np.prod(shape)) and out.flags["C_CONTIGUOUS"]
        st = TcrtStats()
        self._ck(self._lib.tcrt_render_columns_ss(self._h, C.byref(params), ss, x0, x1, out.ctypes.data_as(C.c_void_p),
                                                  C.byref(st)))
        return out.reshape(shape), RenderStats.from_c(st)

    def render_ss_rgb8(self, params: TcrtParams, ss: int, x0: int = 0, x1: Optional[int] = None,
                       out: Optional[np.ndarray] = None):
        """render_ss() quantised to 8 bits on the GPU in the resolve pass (quant8 of the resolved floats); returns
        (array[x1-x0, H, 3] uint8, RenderStats).  The resolved float frame stays on the device as the last render."""
        x1 = params.width if x1 is None else x1
        shape = (x1 - x0, params.height, 3)
        if out is None:
            out = np.empty(shape, dtype=np.uint8)
        assert out.dtype == np.uint8 and out.size == int(np.prod(shape)) and out.flags["C_CONTIGUOUS"]
        st = TcrtStats()
        self._ck(self._lib.tcrt_render_columns_ss_rgb8(self._h, C.byref(params), ss, x0, x1,
                                                       out.ctypes.data_as(C.c_void_p), C.byref(st)))
        return out.reshape(shape), RenderStats.from_c(st)

    def render_ss_device(self, params: TcrtParams, ss: int, x0: int = 0, x1: Optional[int] = None) -> RenderStats:
        """render_ss() left in device memory (download() fetches it), like render_device()."""
        x1 = params.width if x1 is None else x1
        st = TcrtStats()
        self._ck(self._lib.tcrt_render_columns_ss(self._h, C.byref(params), ss, x0, x1, None, C.byref(st)))
        return RenderStats.from_c(st)

    def render_async_ss(self, params: TcrtParams, ss: int, x0: int = 0, x1: Optional[int] = None,
                        out: Optional[np.ndarray] = None) -> int:
        """render_async() of a supersampled frame (into `out`, pinned host memory, when given)."""
        x1 = params.width if x1 is None else x1
        if out is not None:
            assert out.dtype == np.float32 and out.size == (x1 - x0) * params.height * 3 and out.flags["C_CONTIGUOUS"]
        t = C.c_int(-1)
        self._ck(self._lib.tcrt_render_async_ss(self._h, C.byref(params), ss, x0, x1,
                                                out.ctypes.data_as(C.c_void_p) if out is not None else None, C.byref(t)))
        return t.value

    def render_async_ss_rgb8(self, params: TcrtParams, ss: int, x0: int, x1: int, out: np.ndarray) -> int:
        """render_async() of a supersampled 8-bit frame into `out` (uint8, pinned host memory)."""
        assert out.dtype == np.uint8 and out.size == (x1 - x0) * params.height * 3 and out.flags["C_CONTIGUOUS"]
        t = C.c_int(-1)
        self._ck(self._lib.tcrt_render_async_ss_rgb8(self._h, C.byref(params), ss, x0, x1,
                                                     out.ctypes.data_as(C.c_void_p), C.byref(t)))
        return t.value

    def _adaptive(self, fn, dtype, params: TcrtParams, ss: int, contrast: int, x0: int, x1: Optional[int], out, mask,
                  device_only: bool = False):
        x1 = params.width if x1 is None else x1
        shape = (x1 - x0, params.height, 3)
        if out is None and not device_only:
            out = np.empty(shape, dtype=dtype)
        if out is not None:
            assert out.dtype == dtype and out.size == int(np.prod(shape)) and out.flags["C_CONTIGUOUS"]
        if mask is not None:
            assert mask.dtype == np.uint8 and mask.size == (x1 - x0) * params.height and mask.flags["C_CONTIGUOUS"]
        n = C.c_ulonglong(0)
        st = TcrtStats()
        self._ck(fn(self._h, C.byref(params), ss, contrast, x0, x1, out.ctypes.data_as(C.c_void_p) if out is not None else None,
                    mask.ctypes.data_as(C.c_void_p) if mask is not None else None, C.byref(n), C.byref(st)))
        frame = out.reshape(shape) if out is not None else None
        m = mask.reshape(shape[:2]) if mask is not None else None
        return frame, m, int(n.value), RenderStats.from_c(st)

    def render_adaptive(self, params: TcrtParams, ss: int, contrast: int, x0: int = 0, x1: Optional[int] = None,
                        out: Optional[np.ndarray] = None, mask: Optional[np.ndarray] = None):
        """Columns [x0,x1) of the adaptively anti-aliased frame (tcrt_render_columns_adaptive): the render_ss() pixel where
        the plain frame's 3x3 neighbourhood (quant8, max over channels) differs by more than `contrast` (-1: everywhere),
        the render() pixel elsewhere.  `mask` (uint8, (cols, H), optional) receives 1 for every refined pixel.  Returns
        (array[x1-x0, H, 3] float32, mask or None, n_refined, RenderStats).  The frame becomes the last render."""
        return self._adaptive(self._lib.tcrt_render_columns_adaptive, np.float32, params, ss, contrast, x0, x1, out, mask)

    def render_adaptive_rgb8(self, params: TcrtParams, ss: int, contrast: int, x0: int = 0, x1: Optional[int] = None,
                             out: Optional[np.ndarray] = None, mask: Optional[np.ndarray] = None):
        """render_adaptive() quantised to 8 bits on the GPU: (array[x1-x0, H, 3] uint8, mask or None, n_refined,
        RenderStats).  The float frame stays on the device as the last render."""
        return self._adaptive(self._lib.tcrt_render_columns_adaptive_rgb8, np.uint8, params, ss, contrast, x0, x1, out, mask)

    def render_adaptive_device(self, params: TcrtParams, ss: int, contrast: int, x0: int = 0, x1: Optional[int] = None):
        """render_adaptive() left in device memory (download() fetches it): (n_refined, RenderStats)."""
        _, _, n, st = self._adaptive(self._lib.tcrt_render_columns_adaptive, np.float32, params, ss, contrast, x0, x1,
                                     None, None, device_only=True)
        return n, st

    def wait(self, ticket: int) -> RenderStats:
        st = TcrtStats()
        self._ck(self._lib.tcrt_wait(self._h, ticket, C.byref(st)))
        return RenderStats.from_c(st)

    def download(self, out: np.ndarray) -> np.ndarray:
        self._ck(self._lib.tcrt_download(self._h, out.ctypes.data_as(C.c_void_p)))
        return out

    HIT_BUFFERS = (("object", np.int32, ()), ("distance", np.float32, ()), ("normal", np.float32, (3,)))

    def hit_buffers(self, params: TcrtParams, x0: int = 0, x1: Optional[int] = None, out: Optional[dict] = None):
        """What is at each pixel of columns [x0,x1), computed on the GPU (tcrt_hit_buffers): "object" (cols, H) int32, the
        object index of the primary ray's nearest hit or -1; "distance" (cols, H) float32, its distance (far_dist on a
        miss); "normal" (cols, H, 3) float32, its normal ray's direction ((0,0,0) on a miss).  x-major like render().
        `out` maps some of these names to C-contiguous destinations (pinned or pageable); only those are copied back and
        returned.  Returns (dict, RenderStats).  The last render is not touched."""
        x1 = params.width if x1 is None else x1
        cols, h = x1 - x0, params.height
        if out is None:
            out = {name: np.empty((cols, h) + tail, dtype) for name, dtype, tail in self.HIT_BUFFERS}
        ptrs = []
        for name, dtype, tail in self.HIT_BUFFERS:
            a = out.get(name)
            if a is not None:
                assert a.dtype == dtype and a.size == cols * h * int(np.prod(tail)) and a.flags["C_CONTIGUOUS"], name
            ptrs.append(a.ctypes.data_as(C.c_void_p) if a is not None else None)
        st = TcrtStats()
        self._ck(self._lib.tcrt_hit_buffers(self._h, C.byref(params), x0, x1, *ptrs, C.byref(st)))
        res = {name: out[name].reshape((cols, h) + tail) for name, _, tail in self.HIT_BUFFERS if out.get(name) is not None}
        return res, RenderStats.from_c(st)

    def hit_buffers_device(self, params: TcrtParams, x0: int = 0, x1: Optional[int] = None) -> RenderStats:
        """hit_buffers() left in device memory (device_hit_buffers() gives their addresses)."""
        x1 = params.width if x1 is None else x1
        st = TcrtStats()
        self._ck(self._lib.tcrt_hit_buffers(self._h, C.byref(params), x0, x1, None, None, None, C.byref(st)))
        return RenderStats.from_c(st)

    def device_hit_buffers(self, slot: int = 0):
        """Device addresses (object, distance, normal) of device `slot`'s band of the last hit_buffers() call and the
        pixels in it: (int, int, int, n_pixels).  normal holds 3 * n_pixels floats."""
        o, d, n = C.c_void_p(), C.c_void_p(), C.c_void_p()
        cnt = C.c_size_t()
        self._ck(self._lib.tcrt_device_hit_buffers(self._h, slot, C.byref(o), C.byref(d), C.byref(n), C.byref(cnt)))
        return o.value or 0, d.value or 0, n.value or 0, cnt.value

    def pick(self, params: TcrtParams, xs, zs):
        """The hits under pixels (xs[i], zs[i]) of the frame, on device slot 0 (tcrt_pick): (object (n,) int32,
        distance (n,) float32, normal (n, 3) float32), each equal to hit_buffers() at that pixel."""
        xz = np.ascontiguousarray(np.stack([np.asarray(xs, np.int32).ravel(), np.asarray(zs, np.int32).ravel()], axis=1))
        n = xz.shape[0]
        obj = np.empty(n, np.int32)
        dist = np.empty(n, np.float32)
        normal = np.empty((n, 3), np.float32)
        self._ck(self._lib.tcrt_pick(self._h, C.byref(params), n, xz.ctypes.data_as(C.c_void_p), obj.ctypes.data_as(C.c_void_p),
                                     dist.ctypes.data_as(C.c_void_p), normal.ctypes.data_as(C.c_void_p)))
        return obj, dist, normal

    def trace_rays(self, params: TcrtParams, origins, directions, out: Optional[np.ndarray] = None):
        """What caller-supplied rays see (tcrt_trace_rays): origins (n, 3) float32, or (3,) for one origin shared by every
        ray; directions (n, 3) float32, used as a Ray stores them (normalize_like_reference).  Returns (rgb (n, 3) float32,
        n_invalid, RenderStats); an invalid ray's colour is NaN.  `out` (n, 3) float32 may be pinned or pageable."""
        n, o, shared, d = _ray_inputs(origins, directions)
        if out is None:
            out = np.empty((n, 3), np.float32)
        assert out.dtype == np.float32 and out.size == 3 * n and out.flags["C_CONTIGUOUS"], "out: (n, 3) float32"
        bad = C.c_ulonglong(0)
        st = TcrtStats()
        self._ck(self._lib.tcrt_trace_rays(self._h, C.byref(params), n, o.ctypes.data_as(C.c_void_p), shared,
                                           d.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), C.byref(bad),
                                           C.byref(st)))
        return out.reshape(n, 3), int(bad.value), RenderStats.from_c(st)

    def intersect_rays(self, params: TcrtParams, origins, directions, out: Optional[dict] = None):
        """The nearest hits of caller-supplied rays (tcrt_intersect_rays), inputs as in trace_rays: {"object" (n,) int32,
        "distance" (n,) float32, "normal" (n, 3) float32} with the definitions of hit_buffers(); an invalid ray has object
        -2, distance and normal NaN.  `out` maps some of these names to C-contiguous destinations (pinned or pageable);
        only those are computed and returned.  Returns (dict, n_invalid, RenderStats)."""
        n, o, shared, d = _ray_inputs(origins, directions)
        if out is None:
            out = {name: np.empty((n,) + tail, dtype) for name, dtype, tail in self.HIT_BUFFERS}
        ptrs = []
        for name, dtype, tail in self.HIT_BUFFERS:
            a = out.get(name)
            if a is not None:
                assert a.dtype == dtype and a.size == n * int(np.prod(tail)) and a.flags["C_CONTIGUOUS"], name
            ptrs.append(a.ctypes.data_as(C.c_void_p) if a is not None else None)
        bad = C.c_ulonglong(0)
        st = TcrtStats()
        self._ck(self._lib.tcrt_intersect_rays(self._h, C.byref(params), n, o.ctypes.data_as(C.c_void_p), shared,
                                               d.ctypes.data_as(C.c_void_p), *ptrs, C.byref(bad), C.byref(st)))
        res = {name: out[name].reshape((n,) + tail) for name, _, tail in self.HIT_BUFFERS if out.get(name) is not None}
        return res, int(bad.value), RenderStats.from_c(st)

    def render_views(self, params: TcrtParams, cameras, out: Optional[np.ndarray] = None):
        """One scene from a batch of cameras (tcrt_render_views): view v is exactly render(params) after
        set_camera(cameras[v]).  cameras: a sequence of Camera or TcrtCamera.  Returns ((V, W, H, 3) float32, RenderStats);
        the stack is x-major like frames, image rows of view v are a[v].transpose(1, 0, 2)[::-1].  `out` may be pinned or
        pageable.  The ctx camera, the last render and frames in flight are untouched."""
        cams = _camera_table(cameras)
        V, W, H = len(cams), params.width, params.height
        if out is None:
            out = np.empty((V, W, H, 3), np.float32)
        assert out.dtype == np.float32 and out.size == V * W * H * 3 and out.flags["C_CONTIGUOUS"], "out: (V, W, H, 3) float32"
        st = TcrtStats()
        self._ck(self._lib.tcrt_render_views(self._h, C.byref(params), V, C.cast(cams, C.c_void_p),
                                             out.ctypes.data_as(C.c_void_p), None, C.byref(st)))
        return out.reshape(V, W, H, 3), RenderStats.from_c(st)

    def render_views_rgb8(self, params: TcrtParams, cameras, out: Optional[np.ndarray] = None):
        """render_views() quantised on the GPU (tcrt.h's q(c)): ((V, W, H, 3) uint8, RenderStats)."""
        cams = _camera_table(cameras)
        V, W, H = len(cams), params.width, params.height
        if out is None:
            out = np.empty((V, W, H, 3), np.uint8)
        assert out.dtype == np.uint8 and out.size == V * W * H * 3 and out.flags["C_CONTIGUOUS"], "out: (V, W, H, 3) uint8"
        st = TcrtStats()
        self._ck(self._lib.tcrt_render_views(self._h, C.byref(params), V, C.cast(cams, C.c_void_p), None,
                                             out.ctypes.data_as(C.c_void_p), C.byref(st)))
        return out.reshape(V, W, H, 3), RenderStats.from_c(st)

    def render_views_device(self, params: TcrtParams, cameras, rgb: int = 0, rgb8: int = 0, slot: int = 0) -> RenderStats:
        """render_views on device `slot` into device addresses (e.g. torch CUDA tensors' data_ptr()): rgb V*W*H*3 floats,
        rgb8 V*W*H*3 bytes; 0 leaves an output out (not both).  Returns RenderStats."""
        cams = _camera_table(cameras)
        st = TcrtStats()
        self._ck(self._lib.tcrt_render_views_device(self._h, slot, C.byref(params), len(cams), C.cast(cams, C.c_void_p),
                                                    C.c_void_p(rgb or None), C.c_void_p(rgb8 or None), C.byref(st)))
        return RenderStats.from_c(st)

    def trace_rays_device(self, params: TcrtParams, n: int, origins: int, directions: int, rgb: int,
                          shared_origin: bool = False, slot: int = 0):
        """trace_rays on device `slot` with device addresses (e.g. torch CUDA tensors' data_ptr()): origins 3n floats (3
        when shared_origin), directions 3n floats, rgb 3n floats.  The inputs must be complete (synchronise the stream
        that wrote them).  Returns (n_invalid, RenderStats)."""
        bad = C.c_ulonglong(0)
        st = TcrtStats()
        self._ck(self._lib.tcrt_trace_rays_device(self._h, slot, C.byref(params), n, C.c_void_p(origins), int(bool(shared_origin)),
                                                  C.c_void_p(directions), C.c_void_p(rgb), C.byref(bad), C.byref(st)))
        return int(bad.value), RenderStats.from_c(st)

    def intersect_rays_device(self, params: TcrtParams, n: int, origins: int, directions: int, object: int = 0,
                              distance: int = 0, normal: int = 0, shared_origin: bool = False, slot: int = 0):
        """intersect_rays on device `slot` with device addresses as in trace_rays_device; 0 leaves an output out.
        Returns (n_invalid, RenderStats)."""
        bad = C.c_ulonglong(0)
        st = TcrtStats()
        self._ck(self._lib.tcrt_intersect_rays_device(self._h, slot, C.byref(params), n, C.c_void_p(origins),
                                                      int(bool(shared_origin)), C.c_void_p(directions),
                                                      C.c_void_p(object or None), C.c_void_p(distance or None),
                                                      C.c_void_p(normal or None), C.byref(bad), C.byref(st)))
        return int(bad.value), RenderStats.from_c(st)

    def occluded_rays(self, origins, directions, tmax, out: Optional[np.ndarray] = None):
        """The reference's shadow test of caller-supplied rays (tcrt_occluded_rays): origins and directions as in
        trace_rays, tmax (n,) float32 per ray (+inf allowed).  Returns (occluded (n,) uint8, n_invalid, RenderStats): 1 when
        a non-light object is hit at a distance < tmax, 0 if not, 0xFF for an invalid ray or tmax (NaN or <= 0).  `out` (n,)
        uint8 may be pinned or pageable."""
        n, o, shared, d = _ray_inputs(origins, directions)
        t = np.asarray(tmax)
        assert t.dtype == np.float32 and t.shape == (n,) and t.flags["C_CONTIGUOUS"], "tmax: (n,) float32"
        if out is None:
            out = np.empty(n, np.uint8)
        assert out.dtype == np.uint8 and out.size == n and out.flags["C_CONTIGUOUS"], "out: (n,) uint8"
        bad = C.c_ulonglong(0)
        st = TcrtStats()
        self._ck(self._lib.tcrt_occluded_rays(self._h, n, o.ctypes.data_as(C.c_void_p), shared, d.ctypes.data_as(C.c_void_p),
                                              t.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p), C.byref(bad),
                                              C.byref(st)))
        return out.reshape(n), int(bad.value), RenderStats.from_c(st)

    def occluded_lights(self, points, out: Optional[np.ndarray] = None):
        """inShade of caller-supplied points against every light (tcrt_occluded_lights): points (n, 3) float32.  Returns
        (occluded (n, n_lights) uint8, lights in the order of the scene's light_obj, n_invalid (pairs), RenderStats); 0xFF
        marks a point outside the origin rule or one at (within ~1e-19 of) the light.  `out` (n, n_lights) uint8 may be
        pinned or pageable."""
        pts = np.asarray(points)
        assert pts.dtype == np.float32 and pts.ndim == 2 and pts.shape[1] == 3 and pts.flags["C_CONTIGUOUS"], "points: (n, 3) float32"
        n, n_lights = pts.shape[0], getattr(self, "_n_lights", 0)
        if out is None:
            out = np.empty((n, n_lights), np.uint8)
        assert out.dtype == np.uint8 and out.size == n * n_lights and out.flags["C_CONTIGUOUS"], "out: (n, n_lights) uint8"
        bad = C.c_ulonglong(0)
        st = TcrtStats()
        self._ck(self._lib.tcrt_occluded_lights(self._h, n, pts.ctypes.data_as(C.c_void_p), out.ctypes.data_as(C.c_void_p),
                                                C.byref(bad), C.byref(st)))
        return out.reshape(n, n_lights), int(bad.value), RenderStats.from_c(st)

    def occluded_rays_device(self, n: int, origins: int, directions: int, tmax: int, occluded: int,
                             shared_origin: bool = False, slot: int = 0):
        """occluded_rays on device `slot` with device addresses (e.g. torch CUDA tensors' data_ptr()): origins 3n floats
        (3 when shared_origin), directions 3n floats, tmax n floats, occluded n bytes.  The inputs must be complete.
        Returns (n_invalid, RenderStats)."""
        bad = C.c_ulonglong(0)
        st = TcrtStats()
        self._ck(self._lib.tcrt_occluded_rays_device(self._h, slot, n, C.c_void_p(origins), int(bool(shared_origin)),
                                                     C.c_void_p(directions), C.c_void_p(tmax), C.c_void_p(occluded),
                                                     C.byref(bad), C.byref(st)))
        return int(bad.value), RenderStats.from_c(st)

    def occluded_lights_device(self, n: int, points: int, occluded: int, slot: int = 0):
        """occluded_lights on device `slot` with device addresses: points 3n floats, occluded n * n_lights bytes.
        Returns (n_invalid, RenderStats)."""
        bad = C.c_ulonglong(0)
        st = TcrtStats()
        self._ck(self._lib.tcrt_occluded_lights_device(self._h, slot, n, C.c_void_p(points), C.c_void_p(occluded),
                                                       C.byref(bad), C.byref(st)))
        return int(bad.value), RenderStats.from_c(st)

    def balance_columns(self, params: TcrtParams, n_bands: int) -> list[tuple[int, int]]:
        """Cost-balanced column bands of the frame (low-resolution pre-pass on device slot 0):
        [(x0, x1)] * n_bands tiling [0, width).  A measurement: compute it once and share it."""
        b = (C.c_int * (n_bands + 1))()
        self._ck(self._lib.tcrt_balance_columns(self._h, C.byref(params), n_bands, b))
        return [(int(b[i]), int(b[i + 1])) for i in range(n_bands)]

    def flush_l2(self) -> None:
        self._ck(self._lib.tcrt_flush_l2(self._h))

    def selftest_div3(self, n_cases: int, seed: int = 1) -> int:
        """Mismatches of the kernel's shared-reciprocal division against IEEE division."""
        bad = C.c_ulonglong(0)
        self._ck(self._lib.tcrt_selftest_div3(self._h, n_cases, seed, C.byref(bad)))
        return int(bad.value)

    def fp32_peak(self) -> dict:
        """Measured FP32-pipe issue peak of device slot 0 (1e12 lane-instructions/s)."""
        u, f = C.c_double(), C.c_double()
        ms = (C.c_double * 2)()
        self._ck(self._lib.tcrt_fp32_peak(self._h, C.byref(u), C.byref(f), ms))
        return {"unfused_tera_inst": u.value, "fma_tera_inst": f.value, "ms": [ms[0], ms[1]]}

    def txt_size(self) -> int:
        n = C.c_size_t()
        self._ck(self._lib.tcrt_txt_size(self._h, C.byref(n)))
        return n.value

    def format_txt(self, out: Optional[np.ndarray] = None) -> bytes | np.ndarray:
        n = self.txt_size()
        if out is None:
            buf = np.empty(n, dtype=np.uint8)
            got = C.c_size_t()
            self._ck(self._lib.tcrt_format_txt(self._h, buf.ctypes.data_as(C.c_void_p), n, C.byref(got)))
            return buf[: got.value].tobytes()
        got = C.c_size_t()
        self._ck(self._lib.tcrt_format_txt(self._h, out.ctypes.data_as(C.c_void_p), out.nbytes, C.byref(got)))
        return out[: got.value]

    def format_pixels(self, rgb: np.ndarray) -> bytes:
        """The writer's pixel lines for arbitrary float32 pixels (n,3)."""
        rgb = np.ascontiguousarray(rgb, dtype=np.float32).reshape(-1, 3)
        n = rgb.shape[0]
        cap = n * 148 + 16
        buf = np.empty(cap, dtype=np.uint8)
        got = C.c_size_t()
        self._ck(self._lib.tcrt_format_pixels(self._h, rgb.ctypes.data_as(C.c_void_p), n,
                                              buf.ctypes.data_as(C.c_void_p), cap, C.byref(got)))
        return buf[: got.value].tobytes()

    def write_txt(self, params: TcrtParams, path: str, run_time_s: float = 0.0) -> None:
        self._ck(self._lib.tcrt_write_txt(self._h, C.byref(params), path.encode(), run_time_s))

    def write_txt_band(self, params: TcrtParams, path: str, run_time_s: float = 0.0) -> None:
        """The last rendered band's pixel lines at their place in a file made by txt_create (one file from
        several processes, one per GPU)."""
        self._ck(self._lib.tcrt_write_txt_band(self._h, C.byref(params), path.encode(), run_time_s))

    def write_ppm(self, params: TcrtParams, path: str) -> None:
        """The last render as an 8-bit binary PPM (row 0 = top of the image)."""
        self._ck(self._lib.tcrt_write_ppm(self._h, C.byref(params), path.encode()))

    def write_bin(self, params: TcrtParams, path: str) -> None:
        """The last render as raw float32 ("TCRTBIN1" header + pixels[W][H] order)."""
        self._ck(self._lib.tcrt_write_bin(self._h, C.byref(params), path.encode()))

    def update_spheres(self, geom) -> RenderStats:
        """Moving spheres (tcrt_update_spheres): new (centre, radius_squared) rows, (n_spheres, 4) float32 in the order of
        the uploaded scene's sphere_geom (sphere_geom() forms them).  Every later call sees the scene uploaded with these
        spheres (and light spheres' positions at their new centres), bit for bit; the BVH is refitted and the grid
        re-registered on the GPU.  Waits for frames in flight.  Returns RenderStats (render_ms: the update's device time)."""
        g = np.asarray(geom)
        assert g.dtype == np.float32 and g.ndim == 2 and g.shape[1] == 4 and g.flags["C_CONTIGUOUS"], "geom: (n, 4) float32"
        st = TcrtStats()
        self._ck(self._lib.tcrt_update_spheres(self._h, g.ctypes.data_as(C.c_void_p), C.byref(st)))
        return RenderStats.from_c(st)

    def update_spheres_device(self, ptr: int, slot: int = 0) -> RenderStats:
        """update_spheres from device memory of device `slot` (e.g. a torch CUDA tensor's data_ptr(), n_spheres x 4
        float32, 16-byte aligned, complete when called); the other devices of the context get a device-to-device copy.  A
        pointer that is not 16-byte aligned raises TcrtError (TCRT_ERR_INVALID)."""
        st = TcrtStats()
        self._ck(self._lib.tcrt_update_spheres_device(self._h, slot, C.c_void_p(ptr or None), C.byref(st)))
        return RenderStats.from_c(st)

    def update_materials(self, objects, surface=None, material=None, texture=None) -> RenderStats:
        """Material edits (tcrt_update_materials): new rows for the listed objects of the resident scene — surface (n, 4)
        float32 (colour rgb, diffuse), material (n, 4) float32 (specular, reflective, intensity, ignored), texture (n,)
        int32 ids in [-1, n_textures) — each None to leave that part alone (material_rows() forms them).  Every later
        call sees the uploaded scene with those rows replaced, bit for bit.  Which objects are lights and the number of
        textures stay.  Waits for frames in flight.  Returns RenderStats (render_ms: the edit's device time)."""
        obj = np.ascontiguousarray(objects, dtype=np.int32).reshape(-1)
        n = obj.shape[0]

        parts = [None if a is None else np.asarray(a) for a in (surface, material, texture)]
        for a, dtype, shape in zip(parts, (np.float32, np.float32, np.int32), ((n, 4), (n, 4), (n,))):
            assert a is None or (a.dtype == dtype and a.shape == shape and a.flags["C_CONTIGUOUS"]), \
                f"{shape} {np.dtype(dtype).name}"
        ptrs = [None if a is None else C.c_void_p(a.ctypes.data) for a in parts]
        st = TcrtStats()
        self._ck(self._lib.tcrt_update_materials(self._h, n, obj.ctypes.data_as(C.c_void_p), *ptrs, C.byref(st)))
        return RenderStats.from_c(st)

    def update_textures(self, ids, rows) -> RenderStats:
        """Checker edits (tcrt_update_textures): rows (n, 8) float32 (light rgb, width, dark rgb, height) for the texture
        ids `ids` of the resident scene, the layout of the flattened scene's textures."""
        t = np.ascontiguousarray(ids, dtype=np.int32).reshape(-1)
        r = np.asarray(rows)
        assert r.dtype == np.float32 and r.shape == (t.shape[0], 8) and r.flags["C_CONTIGUOUS"], "rows: (n, 8) float32"
        st = TcrtStats()
        self._ck(self._lib.tcrt_update_textures(self._h, t.shape[0], t.ctypes.data_as(C.c_void_p),
                                                r.ctypes.data_as(C.c_void_p), C.byref(st)))
        return RenderStats.from_c(st)

    def update_planes(self, objects, geom, normals, origin) -> RenderStats:
        """Moving planes (tcrt_update_planes): new rows for the listed finite and infinite planes of the resident scene —
        geom (n, 16) float32 (the fin_geom / inf_geom layout by type), normals (n, 8) float32, origin (n, 4) float32 —
        as plane_rows() forms them.  Every later call sees the uploaded scene with those rows replaced, bit for bit; the
        finite-plane BVH and the box clusters follow on the GPU.  Counts, types, lights and materials stay.  Waits for
        frames in flight.  Returns RenderStats (render_ms: the update's device time)."""
        obj = np.ascontiguousarray(objects, dtype=np.int32).reshape(-1)
        n = obj.shape[0]
        parts = [np.asarray(a) for a in (geom, normals, origin)]
        for a, width in zip(parts, (16, 8, 4)):
            assert a.dtype == np.float32 and a.shape == (n, width) and a.flags["C_CONTIGUOUS"], f"({n}, {width}) float32"
        st = TcrtStats()
        self._ck(self._lib.tcrt_update_planes(self._h, n, obj.ctypes.data_as(C.c_void_p),
                                              *[C.c_void_p(a.ctypes.data) for a in parts], C.byref(st)))
        return RenderStats.from_c(st)

    def set_camera(self, cam: TcrtCamera) -> None:
        """Multi-frame mode: new camera, same resident scene."""
        self._ck(self._lib.tcrt_set_camera(self._h, C.byref(cam)))


def txt_header(params: TcrtParams, run_time_s: float) -> bytes:
    buf = C.create_string_buffer(512)
    n = _ffi.load().tcrt_txt_header(C.byref(params), run_time_s, buf, 512)
    if n < 0:
        raise TcrtError(n, "header formatting failed")
    return buf.raw[:n]


def txt_create(params: TcrtParams, path: str, run_time_s: float = 0.0) -> None:
    """Create the .txt with its header and room for width*height 31-byte pixel lines (see write_txt_band)."""
    rc = _ffi.load().tcrt_txt_create(C.byref(params), path.encode(), run_time_s)
    if rc != 0:
        raise TcrtError(rc, _ffi.load().tcrt_last_error(None).decode())


def device_count() -> int:
    return _ffi.load().tcrt_device_count()
