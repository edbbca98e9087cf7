#!/usr/bin/env python
"""Sanitizer substitute (compute-sanitizer is closed on the GPU pool): renders the parity scenes with a -DTCRT_CHECKED
library — every index range-checked, the level stack poisoned and checked for reads of unwritten records — compares
every frame with the oracle bit for bit, and reports the check flags (0 = nothing fired).  Then the same for every
dispatch class of tests/test_kernel_variants.py at the boundary depths of each level stack: band kernels (a tiled and an
untiled frame, a band from an odd column), list kernels (adaptive frames refining every pixel) and hit kernels.  The
flags are read from each translation unit that launches a kernel: render, grid and hits.  Last, a ray batch of valid and
invalid rays on a grid scene and a BVH scene, traced and intersected, against tests/oracle_rays.c, and the occlusion queries
(points against every light, rays with their limits) on a grid scene, BVH scenes and box-cluster scenes against
tests/oracle_occlusion.c.
usage: python -c "from tilecoderaytracer_b200 import build; build.build_lib(defines=('TCRT_CHECKED',), out=LIB)"
       TCRT_LIB=LIB python tools/checked_run.py"""
import ctypes as C
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

from oracle import oracle_py as O  # noqa: E402
from tilecoderaytracer_b200 import _ffi, api  # noqa: E402
import test_kernel_variants as V  # noqa: E402
from test_hit_buffers import assert_hits_equal, primary_hits  # noqa: E402

NAMES = ["pixel store", "level stack index", "BVH stack pointer", "primitive key", "object index", "leaf range", "node index",
         "read of an unwritten level record", "cluster face slot", "queue position"]
lib = _ffi.load()
print("lib:", os.path.basename(_ffi.LIB_PATH), flush=True)
READERS = [lib.tcrt_dev_check_flags, lib.tcrt_dev_grid_check_flags, lib.tcrt_dev_hits_check_flags]
ctx = api.Context([0])
flags = C.c_uint(0)


def fired():
    """Names of the checks that fired since the last call, in any translation unit; resets the flags."""
    bits = 0
    for read in READERS:
        if read(C.byref(flags), 1) != 0:
            raise RuntimeError("cannot read the check flags")
        bits |= flags.value
    return [NAMES[b] for b in range(len(NAMES)) if bits >> b & 1]


def n_bad(img, ref):
    return int((img.view(np.uint32) != ref.view(np.uint32)).any(-1).sum())


def counters_differ(st, cnt):
    return int((st.rays_primary, st.rays_shadow, st.rays_reflect) != (cnt["rays_primary"], cnt["rays_shadow"], cnt["rays_reflect"]))


fired()
bad_total = 0
CASES = [("default", 160, 128, 50), ("boxes:3:14", 128, 96, 12), ("synth256", 160, 128, 10), ("two_mirrors", 96, 80, 50),
         ("synth1024", 160, 128, 50), ("random:24:200", 112, 80, 9), ("random:27:1500", 64, 48, 6), ("random:7:120", 120, 96, 9),
         ("boxes:7:9", 100, 60, 50), ("default", 97, 61, 0), ("default", 64, 48, 200), ("default", 1, 37, 50)]
for name, w, h, d in CASES:
    cam = api.Camera()
    sc = api.Scene().build(name, cam)
    ctx.upload(sc, cam)
    p = api.default_params(w, h, d)
    img, st = ctx.render(p)
    ref, cnt = O.render(sc.flatten(), cam.export(), p)
    bad = n_bad(img, ref)
    f = fired()
    bad_total += bad + len(f)
    print(f"{name:16s} {w}x{h} d{d}: mismatching pixels {bad}, finite {bool(np.isfinite(img).all())}, checks fired: {f or 'none'}", flush=True)

# ---- every dispatch class at the boundary depths of the level stacks --------------------------------------------------------
with tempfile.TemporaryDirectory() as tmp:
    so = os.path.join(tmp, "liboracle_hits.so")
    subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", os.path.join(ROOT, "tests", "oracle_hits.c"),
                    "-o", so, "-lm"], check=True)
    hits_lib = C.CDLL(so)
    hits_lib.tcrt_oracle_primary_hits.restype = C.c_int
    hits_lib.tcrt_oracle_primary_hits.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                  C.c_void_p, C.c_void_p, C.c_void_p]
    for name in V.NAMES:
        s, cam = V.build(name)
        flat, c = s.flatten(), cam.export()
        ctx.upload_flat(flat, c)
        cls = V.dispatch_class(ctx.scene_structures())
        if cls != V.VARIANTS[name][3]:
            print(f"{name}: dispatch class {cls}, expected {V.VARIANTS[name][3]}")
            bad_total += 1
        for d in V.DEPTHS:
            tiled, untiled, (x0, x1) = V.frame_sizes(d)
            bad = 0
            for (w, h), band in ((tiled, (0, tiled[0])), (untiled, (0, untiled[0])), (tiled, (x0, x1))):
                p = api.default_params(w, h, d)
                img, st = ctx.render(p, *band)
                ref, cnt = O.render(flat, c, p, *band)
                bad += n_bad(img, ref) + counters_differ(st, cnt)
            if d in V.LIST_DEPTHS:
                w, h = V.list_frame_size(d)
                p = api.default_params(w, h, d)
                samples, cnt = O.render(flat, c, api.default_params(2 * w, 2 * h, d))
                want = (samples[0::2, 0::2] + samples[0::2, 1::2] + samples[1::2, 0::2] + samples[1::2, 1::2]) / np.float32(4)
                img, _, n, st = ctx.render_adaptive(p, 2, -1)
                bad += n_bad(img, want) + counters_differ(st, cnt) + int(n != w * h)
            f = fired()
            bad_total += bad + len(f)
            print(f"{name:9s} {str(cls):16s} d{d:<3d} cap {V.level_cap(d):3d}: mismatches {bad}, checks fired: {f or 'none'}",
                  flush=True)
        p = api.default_params(27, 17, 8)
        got, _ = ctx.hit_buffers(p)
        try:
            assert_hits_equal(got, primary_hits(hits_lib, flat, c, p), name)
            bad = 0
        except AssertionError as e:
            print(e)
            bad = 1
        f = fired()
        bad_total += bad + len(f)
        print(f"{name:9s} hit buffers 27x17: mismatches {bad}, checks fired: {f or 'none'}", flush=True)

# ---- the placed scenes of tests/test_scene_placement.py: every class moved and rescaled, the lattices at the grid's tightest
# offset, and every far_dist on the grid scene with the camera inside a sphere ---------------------------------------------------
import test_scene_placement as P  # noqa: E402

for pid, name in P.CASES:
    s, flat, c = P.build_placed(pid, name)
    ctx.upload_flat(flat, c)
    bad = int(V.dispatch_class(ctx.scene_structures()) != P.expected_class(pid, name))
    for d in P.DEPTHS:
        p = P.placed_params(pid, name, *P.frame_size(d), d)
        img, st = ctx.render(p)
        ref, cnt = O.render(flat, c, p)
        bad += n_bad(img, ref) + counters_differ(st, cnt)
    f = fired()
    bad_total += bad + len(f)
    print(f"placed {pid:12s} {name:9s} d{P.DEPTHS}: mismatches {bad}, checks fired: {f or 'none'}", flush=True)
s, c = P.inside_sphere_scene()
flat = s.flatten()
ctx.upload_flat(flat, c)
bad = 0
for far in P.FAR_DISTS:
    p = P.far_params(32, 24, 4, far)
    img, st = ctx.render(p)
    ref, cnt = O.render(flat, c, p)
    bad += n_bad(img, ref) + counters_differ(st, cnt)
f = fired()
bad_total += bad + len(f)
print(f"inside_sphere at {len(P.FAR_DISTS)} far_dist values: mismatches {bad}, checks fired: {f or 'none'}", flush=True)

# ---- ray batches: valid and invalid rays mixed, through the render / grid kernels' ray mode and the hit kernel's -----------
import test_ray_batches as R  # noqa: E402

with tempfile.TemporaryDirectory() as tmp:
    so = os.path.join(tmp, "liboracle_rays.so")
    subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", os.path.join(ROOT, "tests", "oracle_rays.c"),
                    "-o", so, "-lm"], check=True)
    rl = C.CDLL(so)
    rl.tcrt_oracle_trace_rays.restype = rl.tcrt_oracle_intersect_rays.restype = C.c_int
    rl.tcrt_oracle_trace_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                          C.POINTER(C.c_ulonglong), C.POINTER(O.OracleCounters)]
    rl.tcrt_oracle_intersect_rays.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_ulonglong)]
    ox, dx, valid = R.crafted_rays()
    for name, grid in (("synth256", True), ("default", False)):
        cam = api.Camera()
        sc = api.Scene().build(name, cam)
        ctx.upload(sc, cam)
        flat = sc.flatten()
        o, d, _ = R.eye_rays(cam.export(), 48, 40, "shuffle")
        o = np.concatenate([o, ox[~valid], o[:7]])
        d = np.concatenate([d, dx[~valid], d[:7]])
        bad = int(ctx.scene_structures()["grid_cells"] > 0) != int(grid)
        for depth in (0, 8, 50):
            p = api.default_params(1, 1, depth)
            got, n_inv, st = ctx.trace_rays(p, o, d)
            want, w_inv, cnt = R.oracle_trace(rl, flat, p, o, d)
            bad += n_bad(got.reshape(-1, 1, 3), want.reshape(-1, 1, 3)) + counters_differ(st, cnt) + int(n_inv != w_inv)
            h, h_inv, _ = ctx.intersect_rays(p, o, d)
            want_h, _ = R.oracle_hits(rl, flat, p, o, d)
            try:
                R.assert_hits_equal(h, want_h, name)
            except AssertionError as e:
                print(e)
                bad += 1
        f = fired()
        bad_total += bad + len(f)
        print(f"ray batch {name:9s} {len(o)} rays ({int((~valid).sum())} invalid), d0/8/50: mismatches {bad}, "
              f"checks fired: {f or 'none'}", flush=True)

# ---- occlusion queries: points against every light and rays with their limits, through the occlusion kernel ---------------
import test_occlusion as Q  # noqa: E402

with tempfile.TemporaryDirectory() as tmp:
    so = os.path.join(tmp, "liboracle_occlusion.so")
    subprocess.run(["gcc", "-std=gnu11", "-O2", "-fPIC", "-shared", "-ffp-contract=off", os.path.join(ROOT, "tests", "oracle_occlusion.c"),
                    "-o", so, "-lm"], check=True)
    ql = C.CDLL(so)
    ull = C.POINTER(C.c_ulonglong)
    ql.tcrt_oracle_occluded_rays.restype = ql.tcrt_oracle_occluded_lights.restype = ql.tcrt_oracle_shadow_origins.restype = C.c_int
    ql.tcrt_oracle_occluded_rays.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, ull, ull]
    ql.tcrt_oracle_occluded_lights.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, ull, ull]
    ql.tcrt_oracle_shadow_origins.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    for name, want_cls in (("synth256", ("grid", 1, 0)), ("random:24:200", ("render", 1, 2)), ("boxes:3:14", ("render", 0, 2)),
                           ("default", ("render", 0, 1)), ("sb1_fm1", ("render", 1, 1))):
        if name in V.VARIANTS:
            sc, cam = V.build(name)
        else:
            cam = api.Camera()
            sc = api.Scene().build(name, cam)
        flat, c = sc.flatten(), cam.export()
        ctx.upload_flat(flat, c)
        bad = int(V.dispatch_class(ctx.scene_structures()) != want_cls)
        rng = np.random.default_rng(5)
        pts = Q.scene_points(ctx, ql, flat, c, rng)
        o, d, t, _, _ = Q.scene_rays(ctx, ql, flat, c, rng)
        o = np.concatenate([o, ox])
        d = np.concatenate([d, dx])
        t = np.concatenate([t, np.full(len(ox), np.float32(np.nan))])
        got, g_bad, st = ctx.occluded_lights(pts)
        want, w_bad, w_tests = Q.oracle_lights(ql, flat, pts)
        bad += int((got != want).any(-1).sum()) + int(g_bad != w_bad) + int(st.rays_shadow != w_tests)
        got, g_bad, st = ctx.occluded_rays(o, d, t)
        want, w_bad, w_tests = Q.oracle_rays(ql, flat, o, d, t)
        bad += int((got != want).sum()) + int(g_bad != w_bad) + int(st.rays_shadow != w_tests)
        f = fired()
        bad_total += bad + len(f)
        print(f"occlusion {name:14s} {str(want_cls):16s} {len(pts)} points x {flat.n_lights} lights, {len(o)} rays: "
              f"mismatches {bad}, checks fired: {f or 'none'}", flush=True)
print("CHECKED_OK" if bad_total == 0 else "CHECKED_FAIL")
