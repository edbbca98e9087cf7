#!/usr/bin/env python
"""Developer tool: moving planes against rebuilding the scene, one process, one GPU.

usage: python tools/e2e_planes.py [--reps N] [--loop N] [--json PATH] [scene ...]

Scenes: the reference's default scene; a room (makeSceneBox, swept through box clusters) with 64 spheres and three lights;
and a tiled box of 6 x 20 x 20 = 2400 finite planes, near the shared-memory staging limit, which gets a finite-plane BVH.
Planes are moved by translation of their rows (normal kept; w = normal . origin, the plane origin and obj_origin shifted),
1 plane and all planes per update, and two ways of getting the moved scene onto the GPU are timed, alternating within each
rep:
  upload   tcrt_upload_scene of the moved scene (moved rows miss the upload cache: the host's sort, BVHs, clusters and grid
           search, then the copy), and an 8x8 depth-0 frame queued behind the copy so that the clock stops when it has
           landed
  update   tcrt_update_planes of the moved planes' rows
Each is a host clock around the blocking call; the update's device time is its render_ms.  Then a loop of --loop frames,
each a move of one wall followed by a 1920x1080 tcrt_render_rgb8 to host memory, against the same loop with an upload of
the moved scene instead: frames per second.  Last, the kernel time (render_ms) of the scene's frame after moving every
plane against after a fresh upload of the moved scene, the median of --reps renders, the two frames checked bit for bit.
Every number is the median (min..max) of --reps reps after one warm-up.  The GPU's name, power limit and max SM clock are
read in the same run.
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
from e2e_update import build_quietly, cell, device_info, frame_ms, summary  # noqa: E402

F32 = np.float32
SCENES = {"default": (1920, 1080, 5), "room": (1920, 1080, 10), "tiled2400": (1920, 1080, 10)}
COUNTS = (1, "all")


def room_scene():
    s = api.Scene()
    for p, inten in (((1.0, 2.0, 6.0), 2.0), ((-3.0, -2.0, 5.0), 1.5), ((4.0, -4.0, 3.0), 1.0)):
        s.addSphere(p, .2).setColor(1, .95, .9).setAsLightSource(inten)
    for k, face in enumerate(s.makeSceneBox((-8, -8, -1), (16, 16, 9))):
        face.setColor(.9, .85, .8).setReflectiveFactor(.5 if k % 2 else 0.0)
    s.addInfinitePlane((0, 0, -1), (0, 0, 1), (1, 0, 0)).setCheckerBoard((1, 1, 1), (.2, .2, .2), 1.5, 1.5)
    for i in range(64):
        s.addSphere((-5 + 1.4 * (i % 8), -5 + 1.4 * (i // 8), 1.0 + .3 * (i % 3)), .45) \
            .setColor(.5 + .4 * (i % 2), .6, .9).setReflectiveFactor(1.0 if i % 4 == 0 else 0.0)
    return s


def tiled_scene(tiles=20):
    s = api.Scene()
    for p, inten in (((1.0, 2.0, 6.0), 2.0), ((-3.0, -2.0, 5.0), 1.5)):
        s.addSphere(p, .2).setColor(1, .95, .9).setAsLightSource(inten)
    lo, hi = np.array([-8.0, -8.0, -1.0]), np.array([8.0, 8.0, 8.0])
    for a in range(3):
        b, c = (a + 1) % 3, (a + 2) % 3
        for side in (lo, hi):
            eb = np.zeros(3)
            ec = np.zeros(3)
            eb[b] = (hi[b] - lo[b]) / tiles
            ec[c] = (hi[c] - lo[c]) / tiles
            base = lo.copy()
            base[a] = side[a]
            for i in range(tiles):
                for j in range(tiles):
                    o = base + i * eb + j * ec
                    s.addFinitePlaneCorners(tuple(o), tuple(o + eb), tuple(o + ec)).setColor(.9, .8 - .1 * a, .7) \
                        .setReflectiveFactor(.5 if (i + j) % 5 == 0 else 0.0)
    for i in range(16):
        s.addSphere((-4 + 2.5 * (i % 4), -4 + 2.5 * (i // 4), 2.0), .8).setReflectiveFactor(1.0)
    return s


def table(flat, name, width, count):
    return np.ctypeslib.as_array(getattr(flat, name), (count * width,)).reshape(count, width)


def plane_objects(flat):
    info = table(flat, "obj_info", 4, flat.n_objects)
    return np.nonzero(info[:, 0] != 0)[0].astype(np.int32)


def shifted(flat, objects, t):
    """Rows of `objects` translated by t: (geom, normals, origin) and the moved flattened scene."""
    geom, normals, origin = api.plane_rows(flat, objects)
    t = np.asarray(t, F32).reshape(-1, 3) * np.ones((len(objects), 1), F32)
    geom[:, 3] += (geom[:, :3] * t).sum(1).astype(F32)   # the row's w is normal . plane origin: the plane moves with it
    geom[:, 12:15] += t
    origin[:, :3] += t
    m = _ffi.TcrtScene.from_buffer_copy(bytes(flat))
    n = flat.n_objects
    info = table(flat, "obj_info", 4, n)
    fin = table(flat, "fin_geom", 16, flat.n_fin_planes).copy() if flat.n_fin_planes else np.zeros((0, 16), F32)
    inf = table(flat, "inf_geom", 16, flat.n_inf_planes).copy() if flat.n_inf_planes else np.zeros((0, 16), F32)
    nr, og = table(flat, "obj_normals", 8, n).copy(), table(flat, "obj_origin", 4, n).copy()
    for i, o in enumerate(objects):
        (fin if info[o, 0] == 1 else inf)[info[o, 1]] = geom[i]
        nr[o], og[o] = normals[i], origin[i]
    m.fin_geom = fin.ctypes.data_as(_ffi.c_float_p) if len(fin) else None
    m.inf_geom = inf.ctypes.data_as(_ffi.c_float_p) if len(inf) else None
    m.obj_normals = nr.ctypes.data_as(_ffi.c_float_p)
    m.obj_origin = og.ctypes.data_as(_ffi.c_float_p)
    m._keep = (fin, inf, nr, og, flat)
    return (geom, normals, origin), m


def run_scene(name, reps, loop):
    w, h, d = SCENES[name]
    cam = api.Camera()
    scene = {"room": room_scene, "tiled2400": tiled_scene}.get(name, lambda: build_quietly(name, cam))()
    flat, c = scene.flatten(), cam.export()
    planes = plane_objects(flat)
    rng = np.random.default_rng(1)
    ctx, ref = api.Context([0]), api.Context([0])
    ctx.upload_flat(flat, c)
    out = {"scene": name, "n_objects": int(flat.n_objects), "n_planes": int(len(planes)),
           "structures": ctx.scene_structures(), "frame": [w, h, d], "updates": []}
    for k in COUNTS:
        k = len(planes) if k == "all" else k
        t_up, t_upd, ms_upd, launches = [], [], [], 0
        for rep in range(reps + 1):
            ctx.upload_flat(flat, c)
            objs = np.sort(rng.choice(planes, k, replace=False)).astype(np.int32)
            rows, m = shifted(flat, objs, rng.normal(0, .05, 3))
            t0 = time.perf_counter()
            ref.upload_flat(m, c)
            ref.render_device(api.default_params(8, 8, 0))   # the upload's copy has landed
            t1 = time.perf_counter()
            st = ctx.update_planes(objs, *rows)
            t2 = time.perf_counter()
            if rep:
                t_up.append(1e3 * (t1 - t0))
                t_upd.append(1e3 * (t2 - t1))
                ms_upd.append(st.render_ms[0])
                launches = st.gpu_launches
        out["updates"].append({"planes": int(k), "upload_ms": summary(t_up), "update_ms": summary(t_upd),
                               "update_gpu_ms": summary(ms_upd), "launches": int(launches)})
    # an update + 1080p rgb8 frame loop against an upload + frame loop: one wall slides back and forth
    p8 = api.default_params(1920, 1080, d)
    buf = api.HostBuffer(1920 * 1080 * 3)
    rgb8 = buf.array(np.uint8, (1920, 1080, 3))
    wall = planes[-1:]
    fps = {}
    for way in ("update", "upload", "update", "upload"):   # alternated; the second pass of each is kept
        target = ctx if way == "update" else ref
        target.upload_flat(flat, c)
        t0 = time.perf_counter()
        for i in range(loop):
            rows, m = shifted(flat, wall, (0, 0, .02 * (i % 8)))
            if way == "update":
                ctx.update_planes(wall, *rows)
            else:
                ref.upload_flat(m, c)
            target.render_rgb8(p8, out=rgb8)
        fps[way] = loop / (time.perf_counter() - t0)
    out["loop_fps"] = fps
    # the frame after moving every plane against after a fresh upload of the moved scene
    rows, m = shifted(flat, planes, rng.normal(0, .05, (len(planes), 3)))
    ctx.upload_flat(flat, c)
    ctx.update_planes(planes, *rows)
    ref.upload_flat(m, c)
    out["structures_after"] = {"update": ctx.scene_structures(), "upload": ref.scene_structures()}
    p = api.default_params(w, h, d)
    a, _ = ctx.render(p)
    a = a.copy()
    b, _ = ref.render(p)
    out["frame_after"] = {"update_ms": frame_ms(ctx, p, reps), "upload_ms": frame_ms(ref, p, reps),
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
        st = r["structures"]
        print(f"\n{name}: {r['n_objects']} objects, {r['n_planes']} planes, finite-plane BVH {st['bvh_finite']}, "
              f"clusters {st['clusters']}, grid cells {st['grid_cells']}; "
              f"frame {r['frame'][0]}x{r['frame'][1]} d{r['frame'][2]}")
        for u in r["updates"]:
            print(f"  {u['planes']:5d} planes  wall ms  upload {cell(u['upload_ms'])}  update {cell(u['update_ms'])}  "
                  f"update GPU ms {cell(u['update_gpu_ms'], 4)}  ({u['launches']} launches)")
        f = r["loop_fps"]
        print(f"  1920x1080 rgb8 frames/s  update + frame {f['update']:.1f}  upload + frame {f['upload']:.1f}")
        f = r["frame_after"]
        print(f"  frame kernel ms  after an update {cell(f['update_ms'])}  after a fresh upload {cell(f['upload_ms'])}  "
              f"bit-identical {f['bit_identical']}")
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as fh:
            json.dump(results, fh, indent=1)


if __name__ == "__main__":
    main()
