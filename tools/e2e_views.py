#!/usr/bin/env python
"""Developer tool: one tcrt_render_views call against a host loop of set_camera + render, one process, one GPU.

usage: python tools/e2e_views.py [--reps N] [--json PATH] [config ...]

For every configuration (default: all of CONFIGS) V views of W x H are rendered four ways, alternating within each rep:
  views_device   one render_views_device call into a torch CUDA buffer
  loop_device    V x (set_camera + render_device): each frame stays in the ctx's device frame buffer
  views_pinned   one render_views call into pinned host memory
  loop_pinned    V x (set_camera + render) into pinned host memory, view after view
Times are a host clock around the whole blocking call or loop, the L2 overwritten (tcrt_flush_l2) before each; the GPU
time is render_ms summed over the calls.  Every number is the median (min..max) of --reps reps after one warm-up rep.  A
correctness line checks that the views equal the loop's frames bit for bit.  The GPU's name, power limit and max SM clock
are read in the same run.
"""
import argparse
import ctypes
import json
import math
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
# name: (scene, V, W, H, depth, camera set)
CONFIGS = {
    "stereo_default_1080p_d50": ("default", 2, 1920, 1080, 50, "stereo"),
    "cube_default_512_d50": ("default", 6, 512, 512, 50, "cube"),
    "turntable_synth256_256_d10": ("synth256", 64, 256, 256, 10, "orbit"),
    "views_two_mirrors_720p_d50": ("two_mirrors", 8, 1280, 720, 50, "moved"),
    "large_synth256_8k_d10": ("synth256", 2, 7680, 4320, 10, "stereo"),
}
CENTRES = {"default": (-1.0, -1.0, 2.5), "synth256": (0.5, 0.5, 0.5), "two_mirrors": (0.0, 3.0, 2.5)}


def device_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        out = [f"nvidia-smi unavailable: {e}"]
    return out


def summary(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


def cell(s, digits=2):
    return f"{s['median']:.{digits}f} ({s['min']:.{digits}f}..{s['max']:.{digits}f})"


def build_scene(name):
    cam = api.Camera()
    sys.stdout.flush()                              # the scene builders print to the C stdout: to stderr, out of the report
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        scene = api.Scene().build(name, cam)
    finally:
        ctypes.CDLL(None).fflush(None)
        os.dup2(saved, 1)
        os.close(saved)
    return scene, cam


def cameras(kind, scene_name, cam, v):
    c = cam.export()
    if kind in ("stereo", "moved"):
        out = []
        for k in range(v):
            m = _ffi.TcrtCamera.from_buffer_copy(bytes(c))
            step = 0.065 * k if kind == "stereo" else 0.05 * k
            for a in range(3):
                m.eye[a] += step * c.horizontal[a]
                m.screen_origin[a] += step * c.horizontal[a]
            out.append(m)
        return out
    centre = CENTRES[scene_name]
    if kind == "cube":
        faces = [((1, 0, 0), (0, 1, 0)), ((-1, 0, 0), (0, -1, 0)), ((0, 1, 0), (-1, 0, 0)), ((0, -1, 0), (1, 0, 0)),
                 ((0, 0, 1), (1, 0, 0)), ((0, 0, -1), (1, 0, 0))]
        out = []
        for o, h in faces[:v]:
            m = api.Camera().aim(tuple(centre[k] + o[k] for k in range(3)), h, o).export()
            m.screen_width = m.screen_height = 2.0
            m.screen_halfwidth = m.screen_halfheight = 1.0
            out.append(m)
        return out
    out = []                                         # orbit
    for k in range(v):
        a = 2 * math.pi * k / v
        so = (centre[0] + 3 * math.cos(a), centre[1] + 3 * math.sin(a), centre[2] + 1)
        out.append(api.Camera().aim(so, (-math.sin(a), math.cos(a), 0.0),
                                    (centre[0] - so[0], centre[1] - so[1], centre[2] - so[2])).export())
    return out


def measure(name, reps):
    import torch

    scene_name, v, w, h, d, kind = CONFIGS[name]
    scene, cam = build_scene(scene_name)
    cams = cameras(kind, scene_name, cam, v)
    p = api.default_params(w, h, d)
    ctx = api.Context([0])
    ctx.upload(scene, cam)
    n = v * w * h * 3
    dev_out = torch.empty(n, dtype=torch.float32, device="cuda:0")
    hb = api.HostBuffer(n * 4)
    pinned = hb.array(F32, (v, w, h, 3))
    torch.cuda.synchronize()

    def views_device():
        return [ctx.render_views_device(p, cams, rgb=dev_out.data_ptr())]

    def loop_device():
        st = []
        for c in cams:
            ctx.set_camera(c)
            st.append(ctx.render_device(p))
        return st

    def views_pinned():
        return [ctx.render_views(p, cams, out=pinned)[1]]

    def loop_pinned():
        st = []
        for k, c in enumerate(cams):
            ctx.set_camera(c)
            st.append(ctx.render(p, out=pinned[k])[1])
        return st

    ways = {"views_device": views_device, "loop_device": loop_device, "views_pinned": views_pinned,
            "loop_pinned": loop_pinned}
    wall = {k: [] for k in ways}
    gpu = {k: [] for k in ways}
    launches = {}
    for rep in range(reps + 1):                      # rep 0 warms up every way
        for key, fn in ways.items():
            ctx.flush_l2()
            t0 = time.perf_counter()
            st = fn()
            ms = (time.perf_counter() - t0) * 1e3
            if rep:
                wall[key].append(ms)
                gpu[key].append(sum(s.render_ms[0] for s in st))
            launches[key] = sum(s.gpu_launches for s in st)
    # correctness: the views of each form against the loop's frames
    views, _ = ctx.render_views(p, cams)
    views = views.copy()
    frames = np.empty_like(views)
    for k, c in enumerate(cams):
        ctx.set_camera(c)
        ctx.render(p, out=frames[k])
    ctx.render_views_device(p, cams, rgb=dev_out.data_ptr())
    dev = dev_out.cpu().numpy().reshape(views.shape)
    correct = bool(np.array_equal(views.view(np.uint32), frames.view(np.uint32))
                   and np.array_equal(dev.view(np.uint32), frames.view(np.uint32)))
    ctx.close()
    del dev_out
    return {"config": name, "scene": scene_name, "views": v, "W": w, "H": h, "depth": d, "cameras": kind,
            "correct": correct, "launches": launches,
            "wall_ms": {k: summary(x) for k, x in wall.items()}, "gpu_ms": {k: summary(x) for k, x in gpu.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("configs", nargs="*", default=list(CONFIGS))
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    info = device_info()
    print("# device:", "; ".join(info))
    print(f"# host clock around whole calls, L2 overwritten before each; median (min..max) of {a.reps} reps after a warm-up")
    results = []
    for name in a.configs:
        r = measure(name, a.reps)
        results.append(r)
        print(f"\n## {name}: {r['views']} x {r['W']}x{r['H']} {r['scene']} d{r['depth']} ({r['cameras']} cameras); "
              f"views bit-identical to the loop's frames: {r['correct']}")
        for key in r["wall_ms"]:
            print(f"{key:13s} wall ms {cell(r['wall_ms'][key])}  gpu ms {cell(r['gpu_ms'][key])}  "
                  f"launches {r['launches'][key]}")
        for form in ("device", "pinned"):
            lw, vw = r["wall_ms"][f"loop_{form}"], r["wall_ms"][f"views_{form}"]
            print(f"{form}: loop / views = {lw['median'] / vw['median']:.3f}x (wall)  "
                  f"[views {vw['min']:.2f}..{vw['max']:.2f}, loop {lw['min']:.2f}..{lw['max']:.2f}]")
    if a.json:
        with open(a.json, "w") as f:
            json.dump({"device": info, "reps": a.reps, "results": results}, f, indent=1)


if __name__ == "__main__":
    main()
