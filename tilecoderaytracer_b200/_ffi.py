"""ctypes declarations for libtcrt.so (include/tcrt.h + include/tcrt_host.h).

The library is the product; there is no Python or CPU implementation of the render path
behind it.  Importing this module fails loudly when the shared library has not been built
(``python -m tilecoderaytracer_b200.build`` / ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# TCRT_LIB: developer override used to A/B kernel variants (tools/quick_perf.py); the product path is the default
LIB_PATH = os.environ.get("TCRT_LIB") or os.path.join(_HERE, "libtcrt.so")

TCRT_MAX_DEVICES = 16
TCRT_OK = 0
TCRT_ERR_INVALID = -1
TCRT_ERR_CUDA = -2
TCRT_ERR_NO_DEVICE = -3
TCRT_ERR_IO = -4
TCRT_ERR_NO_SCENE = -5
TCRT_ERR_NO_FRAME = -6
TCRT_ERR_UNSUPPORTED = -7
TCRT_MAX_DEPTH = 254

c_float_p = C.POINTER(C.c_float)
c_int_p = C.POINTER(C.c_int)


class TcrtScene(C.Structure):
    _fields_ = [
        ("n_objects", C.c_int), ("n_spheres", C.c_int), ("n_fin_planes", C.c_int),
        ("n_inf_planes", C.c_int), ("n_lights", C.c_int), ("n_textures", C.c_int),
        ("sphere_geom", c_float_p), ("sphere_obj", c_int_p),
        ("fin_geom", c_float_p), ("fin_obj", c_int_p),
        ("inf_geom", c_float_p), ("inf_obj", c_int_p),
        ("obj_surface", c_float_p), ("obj_material", c_float_p), ("obj_origin", c_float_p),
        ("obj_normals", c_float_p), ("obj_info", c_int_p),
        ("light_obj", c_int_p), ("textures", c_float_p),
    ]


class TcrtCamera(C.Structure):
    _fields_ = [
        ("eye", C.c_float * 3), ("screen_origin", C.c_float * 3),
        ("horizontal", C.c_float * 3), ("vertical", C.c_float * 3),
        ("screen_width", C.c_float), ("screen_height", C.c_float),
        ("screen_halfwidth", C.c_float), ("screen_halfheight", C.c_float),
    ]


class TcrtParams(C.Structure):
    _fields_ = [
        ("width", C.c_int), ("height", C.c_int), ("max_depth", C.c_int),
        ("shadows_on", C.c_int), ("reflections_on", C.c_int),
        ("null_color", C.c_float * 3), ("far_dist", C.c_float),
    ]


class TcrtStats(C.Structure):
    _fields_ = [
        ("n_devices", C.c_int),
        ("col_begin", C.c_int * TCRT_MAX_DEVICES), ("col_end", C.c_int * TCRT_MAX_DEVICES),
        ("render_ms", C.c_double * TCRT_MAX_DEVICES), ("d2h_ms", C.c_double * TCRT_MAX_DEVICES),
        ("rays_primary", C.c_ulonglong * TCRT_MAX_DEVICES),
        ("rays_shadow", C.c_ulonglong * TCRT_MAX_DEVICES),
        ("rays_reflect", C.c_ulonglong * TCRT_MAX_DEVICES),
        ("gpu_launches", C.c_ulonglong),
    ]


# name -> (restype, argtypes): every symbol include/tcrt.h and include/tcrt_host.h declare
SIGNATURES = {
    # tcrt.h
    "tcrt_abi_version": (C.c_int, []),
    "tcrt_default_params": (None, [C.POINTER(TcrtParams)]),
    "tcrt_device_count": (C.c_int, []),
    "tcrt_create": (C.c_int, [C.POINTER(C.c_void_p), c_int_p, C.c_int]),
    "tcrt_destroy": (None, [C.c_void_p]),
    "tcrt_last_error": (C.c_char_p, [C.c_void_p]),
    "tcrt_alloc_host": (C.c_void_p, [C.c_size_t]),
    "tcrt_free_host": (None, [C.c_void_p]),
    "tcrt_upload_scene": (C.c_int, [C.c_void_p, C.POINTER(TcrtScene), C.POINTER(TcrtCamera)]),
    "tcrt_scene_structures": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "tcrt_plan_scene": (C.c_int, [C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "tcrt_plan_grid_cells": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_float)]),
    "tcrt_plan_dead_paths": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.POINTER(C.c_int)]),
    "tcrt_render": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_void_p, C.POINTER(TcrtStats)]),
    "tcrt_render_columns": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_void_p,
                                      C.POINTER(TcrtStats)]),
    "tcrt_render_device": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.POINTER(TcrtStats)]),
    "tcrt_download": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tcrt_render_async": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]),
    "tcrt_wait": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(TcrtStats)]),
    "tcrt_render_rgb8": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_void_p, C.POINTER(TcrtStats)]),
    "tcrt_render_columns_rgb8": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_void_p,
                                           C.POINTER(TcrtStats)]),
    "tcrt_render_async_rgb8": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_void_p,
                                         C.POINTER(C.c_int)]),
    "tcrt_render_columns_ss": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_int, C.c_void_p,
                                         C.POINTER(TcrtStats)]),
    "tcrt_render_columns_ss_rgb8": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_int, C.c_void_p,
                                              C.POINTER(TcrtStats)]),
    "tcrt_render_async_ss": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_int, C.c_void_p,
                                       C.POINTER(C.c_int)]),
    "tcrt_render_async_ss_rgb8": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_int, C.c_void_p,
                                            C.POINTER(C.c_int)]),
    "tcrt_render_columns_adaptive": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_int, C.c_int,
                                               C.c_void_p, C.c_void_p, C.POINTER(C.c_ulonglong), C.POINTER(TcrtStats)]),
    "tcrt_render_columns_adaptive_rgb8": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_int, C.c_int,
                                                    C.c_void_p, C.c_void_p, C.POINTER(C.c_ulonglong), C.POINTER(TcrtStats)]),
    "tcrt_device_frame": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "tcrt_hit_buffers": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.POINTER(TcrtStats)]),
    "tcrt_device_hit_buffers": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                          C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "tcrt_pick": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tcrt_trace_rays": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_size_t, C.c_void_p, C.c_int, C.c_void_p,
                                  C.c_void_p, C.POINTER(C.c_ulonglong), C.POINTER(TcrtStats)]),
    "tcrt_intersect_rays": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_size_t, C.c_void_p, C.c_int, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_ulonglong), C.POINTER(TcrtStats)]),
    "tcrt_trace_rays_device": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(TcrtParams), C.c_size_t, C.c_void_p, C.c_int,
                                         C.c_void_p, C.c_void_p, C.POINTER(C.c_ulonglong), C.POINTER(TcrtStats)]),
    "tcrt_intersect_rays_device": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(TcrtParams), C.c_size_t, C.c_void_p, C.c_int,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_ulonglong),
                                             C.POINTER(TcrtStats)]),
    "tcrt_occluded_rays": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.POINTER(C.c_ulonglong), C.POINTER(TcrtStats)]),
    "tcrt_occluded_lights": (C.c_int, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.POINTER(C.c_ulonglong),
                                       C.POINTER(TcrtStats)]),
    "tcrt_occluded_rays_device": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.POINTER(C.c_ulonglong), C.POINTER(TcrtStats)]),
    "tcrt_occluded_lights_device": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p, C.c_void_p,
                                              C.POINTER(C.c_ulonglong), C.POINTER(TcrtStats)]),
    "tcrt_render_views": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.POINTER(TcrtStats)]),
    "tcrt_render_views_device": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(TcrtParams), C.c_int, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.POINTER(TcrtStats)]),
    "tcrt_update_spheres": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(TcrtStats)]),
    "tcrt_update_spheres_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(TcrtStats)]),
    "tcrt_update_materials": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.POINTER(TcrtStats)]),
    "tcrt_update_textures": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.POINTER(TcrtStats)]),
    "tcrt_update_planes": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.POINTER(TcrtStats)]),
    "tcrt_flush_l2": (C.c_int, [C.c_void_p]),
    "tcrt_balance_columns": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_int, C.POINTER(C.c_int)]),
    "tcrt_bands_from_costs": (C.c_int, [C.POINTER(C.c_double), C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "tcrt_rebalance_columns": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_double), C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "tcrt_set_camera": (C.c_int, [C.c_void_p, C.POINTER(TcrtCamera)]),
    "tcrt_write_ppm": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_char_p]),
    "tcrt_write_bin": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_char_p]),
    "tcrt_selftest_div3": (C.c_int, [C.c_void_p, C.c_ulonglong, C.c_uint, C.POINTER(C.c_ulonglong)]),
    "tcrt_fp32_peak": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "tcrt_txt_size": (C.c_int, [C.c_void_p, C.POINTER(C.c_size_t)]),
    "tcrt_format_txt": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t)]),
    "tcrt_format_pixels": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                     C.POINTER(C.c_size_t)]),
    "tcrt_txt_header": (C.c_int, [C.POINTER(TcrtParams), C.c_double, C.c_char_p, C.c_size_t]),
    "tcrt_write_txt": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_char_p, C.c_double]),
    "tcrt_txt_create": (C.c_int, [C.POINTER(TcrtParams), C.c_char_p, C.c_double]),
    "tcrt_write_txt_band": (C.c_int, [C.c_void_p, C.POINTER(TcrtParams), C.c_char_p, C.c_double]),
    # tcrt_host.h
    "tcrt_hscene_new": (C.c_void_p, []),
    "tcrt_hscene_free": (None, [C.c_void_p]),
    "tcrt_hcamera_new": (C.c_void_p, []),
    "tcrt_hcamera_free": (None, [C.c_void_p]),
    "tcrt_hcamera_set_two_mirrors": (None, [C.c_void_p]),
    "tcrt_hcamera_export": (None, [C.c_void_p, C.POINTER(TcrtCamera)]),
    "tcrt_hcamera_eye_ray": (None, [C.c_void_p, C.c_float, C.c_float, c_float_p, c_float_p]),
    "tcrt_hcamera_aim": (None, [C.c_void_p, c_float_p, c_float_p, c_float_p]),
    "tcrt_hscene_build": (C.c_int, [C.c_void_p, C.c_void_p, C.c_char_p]),
    "tcrt_hscene_load_text": (C.c_int, [C.c_void_p, C.c_void_p, C.c_char_p, C.c_char_p, C.c_size_t]),
    "tcrt_hscene_add_sphere": (C.c_int, [C.c_void_p, c_float_p, C.c_float]),
    "tcrt_hscene_add_infinite_plane": (C.c_int, [C.c_void_p, c_float_p, c_float_p, c_float_p]),
    "tcrt_hscene_add_finite_plane_corners": (C.c_int, [C.c_void_p, c_float_p, c_float_p, c_float_p]),
    "tcrt_hscene_add_finite_plane_axes": (C.c_int, [C.c_void_p, c_float_p, c_float_p, c_float_p, C.c_float,
                                                    C.c_float]),
    "tcrt_hscene_add_box": (C.c_int, [C.c_void_p, c_float_p, c_float_p]),
    "tcrt_hscene_object_count": (C.c_int, [C.c_void_p]),
    "tcrt_hobj_set_color": (C.c_int, [C.c_void_p, C.c_int, C.c_float, C.c_float, C.c_float]),
    "tcrt_hobj_set_diffuse": (C.c_int, [C.c_void_p, C.c_int, C.c_float]),
    "tcrt_hobj_set_specular": (C.c_int, [C.c_void_p, C.c_int, C.c_float]),
    "tcrt_hobj_set_reflective": (C.c_int, [C.c_void_p, C.c_int, C.c_float]),
    "tcrt_hobj_set_light": (C.c_int, [C.c_void_p, C.c_int, C.c_float]),
    "tcrt_hobj_set_checker": (C.c_int, [C.c_void_p, C.c_int, c_float_p, c_float_p, C.c_float, C.c_float]),
    "tcrt_hscene_flatten": (C.c_int, [C.c_void_p, C.POINTER(TcrtScene)]),
}

_lib = None


def load() -> C.CDLL:
    """Load libtcrt.so and bind every declared symbol.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA library first "
            "(python -m tilecoderaytracer_b200.build, or __graft_entry__.build()). "
            "There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError = ABI mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
