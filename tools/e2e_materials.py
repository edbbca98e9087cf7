#!/usr/bin/env python
"""Developer tool: material edits against rebuilding the scene, one process, one GPU.

usage: python tools/e2e_materials.py [--reps N] [--loop N] [--json PATH] [scene ...]

For every scene (default: synth256, synth1024, lattice3840 and two_mirrors, as in tools/e2e_update.py) new colours and
factors are given to 1, 64 and all objects, and two ways of getting the edited scene onto the GPU are timed, alternating
within each rep:
  upload   tcrt_upload_scene of the edited scene (an edited colour misses the upload cache: the host's sort, BVH,
           clusters and grid search, then the copy), and an 8x8 depth-0 frame queued behind the copy so that the clock
           stops when it has landed
  edit     tcrt_update_materials of the edited objects' rows
Each is a host clock around the blocking call; the edit's device time is its render_ms.  Then a loop of --loop frames,
each an edit of one light's intensity followed by a 1920x1080 tcrt_render_rgb8 to host memory, against the same loop with
an upload of the edited scene instead of the edit: frames per second.  Last, the kernel time (render_ms) of the scene's
frame after an edit of every object against after a fresh upload of the edited scene, the median of --reps renders, the
two frames checked bit for bit.  Every number is the median (min..max) of --reps reps after one warm-up.  The GPU's name,
power limit and max SM clock are read in the same run.
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402

from tilecoderaytracer_b200 import _ffi, api  # noqa: E402
from e2e_update import SCENES, build_quietly, cell, device_info, frame_ms, lattice3840, summary  # noqa: E402

F32 = np.float32
COUNTS = (1, 64, "all")


def table(flat, name, width):
    n = flat.n_objects
    return np.ctypeslib.as_array(getattr(flat, name), (n * width,)).reshape(n, width)


def edited_flat(flat, objects, surface, material):
    """The flattened scene with the surface and material rows of `objects` replaced."""
    m = _ffi.TcrtScene.from_buffer_copy(bytes(flat))
    s, mt = table(flat, "obj_surface", 4).copy(), table(flat, "obj_material", 4).copy()
    s[objects], mt[objects] = surface, material
    m.obj_surface = s.ctypes.data_as(_ffi.c_float_p)
    m.obj_material = mt.ctypes.data_as(_ffi.c_float_p)
    m._keep = (s, mt, flat)
    return m


def recolour(flat, objects, rng):
    """New colours, diffuse and specular factors for `objects`; their reflective factors and intensities stay."""
    s, m, _ = api.material_rows(flat, objects)
    s[:] = rng.uniform(0.1, 1.0, s.shape).astype(F32)
    m[:, 0] = rng.uniform(0.0, 1.0, len(m)).astype(F32)
    return s, m


def run_scene(name, reps, loop):
    w, h, d = SCENES[name]
    cam = api.Camera()
    scene = lattice3840() if name == "lattice3840" else build_quietly(name, cam)
    flat, c = scene.flatten(), cam.export()
    n = flat.n_objects
    rng = np.random.default_rng(1)
    ctx, ref = api.Context([0]), api.Context([0])
    ctx.upload_flat(flat, c)
    out = {"scene": name, "n_objects": int(n), "structures": ctx.scene_structures(), "frame": [w, h, d], "edits": []}
    for k in COUNTS:
        k = n if k == "all" else min(k, n)
        t_up, t_edit, ms_edit = [], [], []
        for rep in range(reps + 1):
            objs = np.sort(rng.choice(n, k, replace=False)).astype(np.int32)
            s, m = recolour(flat, objs, rng)
            e = edited_flat(flat, objs, s, m)
            t0 = time.perf_counter()
            ref.upload_flat(e, c)
            ref.render_device(api.default_params(8, 8, 0))   # the upload's copy has landed
            t1 = time.perf_counter()
            st = ctx.update_materials(objs, s, m)
            t2 = time.perf_counter()
            if rep:
                t_up.append(1e3 * (t1 - t0))
                t_edit.append(1e3 * (t2 - t1))
                ms_edit.append(st.render_ms[0])
        out["edits"].append({"objects": int(k), "upload_ms": summary(t_up), "edit_ms": summary(t_edit),
                             "edit_gpu_ms": summary(ms_edit)})
    # an edit + 1080p rgb8 frame loop against an upload + frame loop
    p8 = api.default_params(1920, 1080, d)
    buf = api.HostBuffer(1920 * 1080 * 3)
    rgb8 = buf.array(np.uint8, (1920, 1080, 3))
    info = table(flat, "obj_info", 4)
    light = np.array([int(np.nonzero(info[:, 2])[0][0])], np.int32)
    fps = {}
    for way in ("edit", "upload", "edit", "upload"):   # alternated; the second pass of each is kept
        target = ctx if way == "edit" else ref
        target.upload_flat(flat, c)
        t0 = time.perf_counter()
        for i in range(loop):
            s, m, _ = api.material_rows(flat, light)
            m[:, 2] = F32(0.5 + (i % 8) / 8)
            if way == "edit":
                ctx.update_materials(light, s, m)
            else:
                ref.upload_flat(edited_flat(flat, light, s, m), c)
            target.render_rgb8(p8, out=rgb8)
        fps[way] = loop / (time.perf_counter() - t0)
    out["loop_fps"] = fps
    # the frame after an edit of every object against after a fresh upload of the edited scene
    objs = np.arange(n, dtype=np.int32)
    s, m = recolour(flat, objs, rng)
    ctx.upload_flat(flat, c)
    ctx.update_materials(objs, s, m)
    ref.upload_flat(edited_flat(flat, objs, s, m), c)
    p = api.default_params(w, h, d)
    a, _ = ctx.render(p)
    a = a.copy()
    b, _ = ref.render(p)
    out["frame_after"] = {"edit_ms": frame_ms(ctx, p, reps), "upload_ms": frame_ms(ref, p, reps),
                          "bit_identical": bool((a.view(np.uint32) == b.view(np.uint32)).all())}
    ctx.close()
    ref.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--loop", type=int, default=30)
    ap.add_argument("--json", default=None)
    ap.add_argument("scenes", nargs="*", default=list(SCENES))
    a = ap.parse_args()
    info = device_info()
    print("GPU (name, power limit, max SM clock):", "; ".join(info))
    results = {"gpu": info, "reps": a.reps, "loop": a.loop, "scenes": []}
    for name in a.scenes:
        r = run_scene(name, a.reps, a.loop)
        results["scenes"].append(r)
        print(f"\n{name}: {r['n_objects']} objects, grid cells {r['structures']['grid_cells']}, "
              f"BVH spheres {r['structures']['bvh_spheres']}; frame {r['frame'][0]}x{r['frame'][1]} d{r['frame'][2]}")
        for e in r["edits"]:
            print(f"  {e['objects']:5d} objects  wall ms  upload {cell(e['upload_ms'])}  edit {cell(e['edit_ms'])}  "
                  f"edit GPU ms {cell(e['edit_gpu_ms'], 4)}")
        f = r["loop_fps"]
        print(f"  1920x1080 rgb8 frames/s  edit + frame {f['edit']:.1f}  upload + frame {f['upload']:.1f}")
        f = r["frame_after"]
        print(f"  frame kernel ms  after an edit {cell(f['edit_ms'])}  after a fresh upload {cell(f['upload_ms'])}  "
              f"bit-identical {f['bit_identical']}")
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as fh:
            json.dump(results, fh, indent=1)


if __name__ == "__main__":
    main()
