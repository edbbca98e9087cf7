#!/usr/bin/env python
"""Developer tool: moving spheres against rebuilding the scene, one process, one GPU.

usage: python tools/e2e_update.py [--reps N] [--json PATH] [scene ...]

For every scene (default: synth256, synth1024, lattice3840 — a 16 x 16 x 15 lattice of spheres in the unit cube, built
here, the largest lattice of that kind under the Scene's 4095-object cap — and two_mirrors) the spheres are jittered
inwards (inward_jitter: the grid is kept) and three ways of getting the moved scene onto the GPU are timed, alternating
within each rep:
  upload          tcrt_upload_scene of the moved scene (the host's sort, BVH, clusters and grid search, then the copy),
                  and an 8x8 depth-0 frame queued behind the copy so that the clock stops when it has landed
  update_host     tcrt_update_spheres from a numpy array
  update_device   tcrt_update_spheres_device from a torch CUDA tensor
Each is a host clock around the blocking call (every one ends in a device synchronise); the update's device time is its
render_ms.  Then the frame after an update against the frame after a fresh upload of the same geometry, for one small
jitter and after 100 drift steps applied to the already-updated scene: kernel time (render_ms) of the scene's
BASELINE-sized frame, the median of --reps renders, each frame checked bit for bit against the fresh upload's; and once
for a jitter that may move the outermost spheres outwards, which drops the grid.  Every
number is the median (min..max) of --reps reps after one warm-up.  The GPU's name, power limit and max SM clock are read
in the same run.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True
import numpy as np  # noqa: E402

from tilecoderaytracer_b200 import _ffi, api  # noqa: E402

F32 = np.float32
# scene: (W, H, depth) of the frame that is timed
SCENES = {
    "synth256": (1920, 1080, 10),
    "synth1024": (3840, 2160, 50),
    "lattice3840": (1920, 1080, 10),
    "two_mirrors": (1920, 1080, 50),
}


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        out = [f"nvidia-smi unavailable: {e}"]
    return out


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


def cell(s, digits=3):
    return f"{s['median']:.{digits}f} ({s['min']:.{digits}f}..{s['max']:.{digits}f})"


def geom_of(flat):
    n = flat.n_spheres
    return np.ctypeslib.as_array(flat.sphere_geom, (n * 4,)).reshape(n, 4).astype(F32)


def moved_flat(flat, geom):
    """The flattened scene with sphere_geom = geom and each sphere's obj_origin row at its new centre."""
    m = _ffi.TcrtScene.from_buffer_copy(bytes(flat))
    g = np.ascontiguousarray(geom, F32).copy()
    origin = np.ctypeslib.as_array(flat.obj_origin, (flat.n_objects * 4,)).reshape(-1, 4).copy()
    objs = np.ctypeslib.as_array(flat.sphere_obj, (flat.n_spheres,))
    origin[objs, :3] = g[:, :3]
    m.sphere_geom = g.ctypes.data_as(_ffi.c_float_p)
    m.obj_origin = origin.ctypes.data_as(_ffi.c_float_p)
    m._keep = (g, origin, flat)
    return m


def spacing(geom):
    c = geom[:, :3].astype(np.float64)
    best = np.full(len(c), np.inf)
    for i in range(0, len(c), 512):   # nearest neighbour in blocks: 4k x 4k distances would be 128 MB
        d = ((c[i:i + 512, None, :] - c[None, :, :]) ** 2).sum(-1)
        d[np.arange(d.shape[0]), np.arange(i, i + d.shape[0])] = np.inf
        best[i:i + 512] = np.sqrt(d.min(1))
    return float(np.median(best))


def lattice3840():
    """16 x 16 x 15 spheres of radius 0.4 / 16 on a 1/16 lattice in the unit cube (where synth256's are), two light
    spheres."""
    s = api.Scene()
    for k in range(15):
        for j in range(16):
            for i in range(16):
                s.addSphere(((i + .5) / 16, (j + .5) / 16, (k + .5) / 16), .4 / 16) \
                    .setColor(.4 + .5 * (i % 2), .5 + .4 * (j % 2), .9 - .5 * (k % 2)).setReflectiveFactor(.5)
    s.addSphere((-2.0, -3.0, 3.0), .2).setAsLightSource(1.5)
    s.addSphere((2.5, -1.0, 2.0), .2).setAsLightSource(1.0)
    return s


def light_spheres(flat):
    info = np.ctypeslib.as_array(flat.obj_info, (flat.n_objects * 4,)).reshape(-1, 4)
    objs = np.ctypeslib.as_array(flat.sphere_obj, (flat.n_spheres,))
    return np.nonzero(info[objs, 2])[0]


def inward_jitter(geom, rng, scale, lights):
    """Centres jittered by `scale` (standard deviation); a sphere within half the spacing of the bounding box of the
    moving centres moves only inwards along that axis, so that the grid, whose box the upload fits tightly around the
    spheres, is kept.  The light spheres stay."""
    moving = ~np.isin(np.arange(len(geom)), lights)
    s = spacing(geom[moving])
    lo, hi = geom[moving, :3].min(0), geom[moving, :3].max(0)
    d = rng.normal(0.0, scale, geom[:, :3].shape).astype(F32)
    d = np.where(geom[:, :3] < lo + 0.5 * s, np.abs(d), d)
    d = np.where(geom[:, :3] > hi - 0.5 * s, -np.abs(d), d)
    d[~moving] = 0
    g = geom.copy()
    g[:, :3] += d
    return g


def build_quietly(name, cam):
    """The named scene; the C++ Scene builder prints "ObjectCount: ..." for SCENE 2, kept out of the recorded output."""
    sys.stdout.flush()
    saved = os.dup(1)
    with open(os.devnull, "w") as null:
        os.dup2(null.fileno(), 1)
        try:
            return api.Scene().build(name, cam)
        finally:
            os.dup2(saved, 1)
            os.close(saved)


def frame_ms(ctx, p, reps):
    ctx.render_device(p)
    return summary([ctx.render_device(p).render_ms[0] for _ in range(reps)])


def run_scene(name, reps, torch):
    w, h, d = SCENES[name]
    cam = api.Camera()
    scene = lattice3840() if name == "lattice3840" else build_quietly(name, cam)
    flat, c = scene.flatten(), cam.export()
    g0 = geom_of(flat)
    lights = light_spheres(flat)
    s = spacing(np.delete(g0, lights, 0))
    rng = np.random.default_rng(1)
    ctx, ref = api.Context([0]), api.Context([0])
    ctx.upload_flat(flat, c)
    structures = ctx.scene_structures()
    p = api.default_params(w, h, d)
    t_up, t_host, t_dev, ms_host, ms_dev = [], [], [], [], []
    for rep in range(reps + 1):
        g = inward_jitter(g0, rng, 0.02 * s, lights)
        m = moved_flat(flat, g)
        tg = torch.from_numpy(g).cuda()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ref.upload_flat(m, c)
        ref.render_device(api.default_params(8, 8, 0))   # the upload's copy has landed
        t1 = time.perf_counter()
        st_h = ctx.update_spheres(g)
        t2 = time.perf_counter()
        st_d = ctx.update_spheres_device(tg.data_ptr())
        t3 = time.perf_counter()
        if rep:
            t_up.append(1e3 * (t1 - t0))
            t_host.append(1e3 * (t2 - t1))
            t_dev.append(1e3 * (t3 - t2))
            ms_host.append(st_h.render_ms[0])
            ms_dev.append(st_d.render_ms[0])
    # frames: small jitter, then 100 drift steps
    out = {"scene": name, "n_spheres": int(flat.n_spheres), "structures": structures, "frame": [w, h, d],
           "upload_ms": summary(t_up), "update_host_ms": summary(t_host), "update_device_ms": summary(t_dev),
           "update_host_gpu_ms": summary(ms_host), "update_device_gpu_ms": summary(ms_dev)}
    g = g0.copy()
    ctx.upload_flat(flat, c)
    for step in range(1, 101):
        g = inward_jitter(g, rng, (0.02 if step == 1 else 0.005) * s, lights)
        ctx.update_spheres(g)
        if step in (1, 100):
            m = moved_flat(flat, g)
            ref.upload_flat(m, c)
            a, _ = ctx.render(p)
            b, _ = ref.render(p)
            same = bool((a.view(np.uint32) == b.view(np.uint32)).all())
            key = "jitter" if step == 1 else "drift100"
            out[key] = {"after_update_ms": frame_ms(ctx, p, reps), "after_upload_ms": frame_ms(ref, p, reps),
                        "bit_identical": same, "grid_cells_update": ctx.scene_structures()["grid_cells"],
                        "grid_cells_upload": ref.scene_structures()["grid_cells"]}
    g = g0.copy()
    g[:, :3] += rng.normal(0.0, 0.02 * s, g[:, :3].shape).astype(F32)
    g[lights] = g0[lights]
    ctx.upload_flat(flat, c)
    ctx.update_spheres(g)
    ref.upload_flat(moved_flat(flat, g), c)
    a, _ = ctx.render(p)
    b, _ = ref.render(p)
    out["outward"] = {"after_update_ms": frame_ms(ctx, p, reps), "after_upload_ms": frame_ms(ref, p, reps),
                      "bit_identical": bool((a.view(np.uint32) == b.view(np.uint32)).all()),
                      "grid_cells_update": ctx.scene_structures()["grid_cells"],
                      "grid_cells_upload": ref.scene_structures()["grid_cells"]}
    ctx.close()
    ref.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--json", default=None)
    ap.add_argument("scenes", nargs="*", default=list(SCENES))
    a = ap.parse_args()
    import torch

    info = device_info()
    print("GPU (name, power limit, max SM clock):", "; ".join(info))
    results = {"gpu": info, "reps": a.reps, "scenes": []}
    for name in a.scenes:
        r = run_scene(name, a.reps, torch)
        results["scenes"].append(r)
        print(f"\n{name}: {r['n_spheres']} spheres, grid cells {r['structures']['grid_cells']}, "
              f"BVH spheres {r['structures']['bvh_spheres']}; frame {r['frame'][0]}x{r['frame'][1]} d{r['frame'][2]}")
        print(f"  wall ms  upload {cell(r['upload_ms'])}  update host {cell(r['update_host_ms'])}  "
              f"update device {cell(r['update_device_ms'])}")
        print(f"  update GPU ms  host form {cell(r['update_host_gpu_ms'])}  device form {cell(r['update_device_gpu_ms'])}")
        for key in ("jitter", "drift100", "outward"):
            f = r[key]
            print(f"  frame kernel ms after {key}: update {cell(f['after_update_ms'])}  fresh upload "
                  f"{cell(f['after_upload_ms'])}  bit-identical {f['bit_identical']}  grid cells "
                  f"{f['grid_cells_update']} / {f['grid_cells_upload']}")
    if a.json:
        os.makedirs(os.path.dirname(os.path.abspath(a.json)), exist_ok=True)
        with open(a.json, "w") as fh:
            json.dump(results, fh, indent=1)


if __name__ == "__main__":
    main()
